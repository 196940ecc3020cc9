// stream.cu -- streaming ingest (SURVEY 8f rank 3; reference README.md:23 "Decisions" 3 wants streaming,
// src/lib.rs:64-65 mmaps the whole file): csv of ANY size -> index, in bounded device and pinned memory.
//
//   reader (callback, or a pool of threads pread()ing a file)  ->  pinned input ring
//   -> cudaMemcpyAsync H2D -> fused index kernel, chained to the previous chunk through a device cell that
//      carries the quote parity (no host round trip between launches)
//   -> D2H of the chunk's index segment on a second stream -> sink callback (or the caller's array)
//
// Chunk c+1 is read and uploaded while chunk c is indexed and chunk c-1 comes down; a chunk's segment
// buffer on the device holds the worst case (one entry per byte), so no launch can overflow, and the
// pinned output ring is drained in pieces when a chunk is denser than the ring slot.
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>

#include "ctx.h"
#include "slice_pool.h"

using namespace csvb200;

namespace {

constexpr int kSlots = 3;                        // ring depth: read / index / drain
constexpr size_t kDefaultChunk = 16u << 20;
constexpr size_t kMinChunk = 64u << 10;

struct Slot {
    uint8_t* h_in = nullptr;       // pinned
    uint64_t* h_out = nullptr;     // pinned, out_cap entries
    uint8_t* d_in = nullptr;
    uint64_t* d_seg = nullptr;     // chunk + 2 entries: the worst case (one entry per byte) + sentinel
    cudaEvent_t k_done = nullptr;  // kernel of the chunk in this slot (it writes its count to the pinned cell)
    cudaEvent_t d_done = nullptr;  // last D2H out of d_seg
    size_t bytes = 0;              // bytes of the chunk in flight
    uint64_t offset = 0;           // global byte offset of the chunk
    size_t cell = 0;
    bool busy = false;
};

struct Pipeline {
    csvb200_ctx* ctx = nullptr;
    size_t chunk = 0, out_cap = 0;
    Slot slot[kSlots];
    size_t cells0 = 0;             // kSlots + 1 consecutive result cells; cell of chunk c = cells0 + c % (kSlots + 1)
    uint64_t next_slot_global = 0; // global index slot of the next entry to hand to the sink
    uint64_t total_bytes = 0;
    uint32_t chunks = 0;
    int end_parity = 0;

    ~Pipeline()
    {
        if (!ctx) return;
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->copy_stream);
        for (Slot& s : slot) {
            if (s.d_in) cudaFreeAsync(s.d_in, ctx->stream);
            if (s.d_seg) cudaFreeAsync(s.d_seg, ctx->stream);
            if (s.k_done) cudaEventDestroy(s.k_done);
            if (s.d_done) cudaEventDestroy(s.d_done);
        }
        cell_release(ctx, cells0, kSlots + 1);
        cudaGetLastError();
    }

    int init(csvb200_ctx* c, size_t chunk_bytes)
    {
        ctx = c;
        chunk = std::max(kMinChunk, chunk_bytes ? chunk_bytes : kDefaultChunk);
        chunk = (chunk + 127) & ~size_t(127);          // chunk boundaries stay 128-byte aligned (TMA rows)
        out_cap = chunk / 2 + 4096;                    // entries per pinned output slot (4 x the chunk's bytes)
        CU_TRY(ctx, cudaSetDevice(ctx->device));
        cells0 = cell_alloc(ctx, kSlots + 1);   // held until the pipeline object dies
        if (cells0 == SIZE_MAX) return fail(ctx, CSVB200_ERR_OOM, "no free result cells (4095 live index objects)");
        static_assert(kSlots == 3, "the context caches three ring slots");
        if (ctx->stream_chunk != chunk || ctx->stream_out_cap != out_cap) {   // (re)build the context's pinned rings
            for (int i = 0; i < kSlots; ++i) {
                if (ctx->h_stream_in[i]) cudaFreeHost(ctx->h_stream_in[i]);
                if (ctx->h_stream_out[i]) cudaFreeHost(ctx->h_stream_out[i]);
                ctx->h_stream_in[i] = nullptr;
                ctx->h_stream_out[i] = nullptr;
            }
            ctx->stream_chunk = ctx->stream_out_cap = 0;
            for (int i = 0; i < kSlots; ++i) {
                CU_TRY(ctx, cudaHostAlloc((void**)&ctx->h_stream_in[i], chunk, cudaHostAllocDefault));
                CU_TRY(ctx, cudaHostAlloc((void**)&ctx->h_stream_out[i], out_cap * sizeof(uint64_t), cudaHostAllocDefault));
            }
            ctx->stream_chunk = chunk;
            ctx->stream_out_cap = out_cap;
        }
        int si = 0;
        for (Slot& s : slot) {
            s.h_in = ctx->h_stream_in[si];
            s.h_out = ctx->h_stream_out[si];
            ++si;
            CU_TRY(ctx, pool_malloc((void**)&s.d_in, chunk + 16, ctx->stream));
            CU_TRY(ctx, pool_malloc((void**)&s.d_seg, (chunk + 2) * sizeof(uint64_t), ctx->stream));
            CU_TRY(ctx, cudaEventCreateWithFlags(&s.k_done, cudaEventDisableTiming));
            CU_TRY(ctx, cudaEventCreateWithFlags(&s.d_done, cudaEventDisableTiming));
        }
        // carry into chunk 0: {0, parity 0}
        CU_TRY(ctx, cudaMemsetAsync(ctx->d_cells + (cells0 + kSlots) * kCellWords, 0, kCellWords * sizeof(uint64_t), ctx->stream));
        return CSVB200_OK;
    }

    size_t cell_of(uint32_t c) const { return cells0 + c % (kSlots + 1); }

    // enqueue H2D + kernel of the chunk sitting in slot s (s.bytes > 0)
    int launch(Slot& s)
    {
        const uint32_t c = chunks;
        s.offset = total_bytes;
        s.cell = cell_of(c);
        const size_t prev_cell = c == 0 ? cells0 + kSlots : cell_of(c - 1);
        cudaStream_t st = ctx->stream;
        CU_TRY(ctx, cudaStreamWaitEvent(st, s.d_done, 0));   // the previous segment in this slot has left d_seg
        CU_TRY(ctx, cudaMemcpyAsync(s.d_in, s.h_in, s.bytes, cudaMemcpyHostToDevice, st));
        BuildParams p{};
        p.in = s.d_in;
        p.n = s.bytes;
        p.index = s.d_seg;
        p.cap = chunk + 2;
        p.out_base = c == 0 ? 1 : 0;
        p.pos_bias = s.offset;
        p.carry = ctx->d_cells + prev_cell * kCellWords;
        p.carry_parity_only = 1;
        p.write_sentinel = c == 0 ? 1u : 0u;     // sentinel (src/reader.rs:216)
        const int rc = launch_build(ctx, p, s.cell, st);
        if (rc) return rc;
        CU_TRY(ctx, cudaEventRecord(s.k_done, st));
        s.busy = true;
        total_bytes += s.bytes;
        ++chunks;
        return CSVB200_OK;
    }

    // wait for the chunk in slot s, bring its segment down (in pieces of the pinned slot) and hand it on.
    // direct_dst != nullptr: the caller's array is pinned, entries go straight into it.
    int drain(Slot& s, const std::function<int(const uint64_t*, size_t, uint64_t)>& sink, uint64_t* direct_dst,
              size_t direct_cap, bool* dst_small)
    {
        if (!s.busy) return CSVB200_OK;
        CU_TRY(ctx, cudaEventSynchronize(s.k_done));
        const uint64_t* h_cell = ctx->h_cells + s.cell * kCellWords;
        const size_t count = (size_t)h_cell[0] + (s.offset == 0 ? 1 : 0);   // + sentinel in the first chunk
        end_parity = (int)(h_cell[1] & 1u);
        cudaStream_t sd = ctx->copy_stream;
        CU_TRY(ctx, cudaStreamWaitEvent(sd, s.k_done, 0));
        if (direct_dst) {
            if (next_slot_global + count > direct_cap) {
                *dst_small = true;
            } else if (count) {
                CU_TRY(ctx, cudaMemcpyAsync(direct_dst + next_slot_global, s.d_seg, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, sd));
            }
            CU_TRY(ctx, cudaEventRecord(s.d_done, sd));
            next_slot_global += count;
        } else {
            for (size_t off = 0; off < count; off += out_cap) {
                const size_t len = std::min(out_cap, count - off);
                CU_TRY(ctx, cudaMemcpyAsync(s.h_out, s.d_seg + off, len * sizeof(uint64_t), cudaMemcpyDeviceToHost, sd));
                CU_TRY(ctx, cudaStreamSynchronize(sd));
                if (sink(s.h_out, len, next_slot_global) != 0) return fail(ctx, CSVB200_ERR_IO, "index sink reported an error");
                next_slot_global += len;
            }
            CU_TRY(ctx, cudaEventRecord(s.d_done, sd));
        }
        s.busy = false;
        return CSVB200_OK;
    }
};

using ReadFn = std::function<long long(uint8_t*, size_t)>;   // fills up to cap bytes, < cap only at the end, < 0 = error
using SinkFn = std::function<int(const uint64_t*, size_t, uint64_t)>;

int run_pipeline(csvb200_ctx* ctx, size_t chunk_bytes, const ReadFn& read, const SinkFn& sink, uint64_t* direct_dst,
                 size_t direct_cap, csvb200_stream_stats* stats)
{
    const auto t0 = std::chrono::steady_clock::now();
    Pipeline pl;
    int rc = pl.init(ctx, chunk_bytes);
    if (rc) return rc;
    bool dst_small = false, eof = false;
    uint32_t head = 0, tail = 0;   // chunks launched / drained
    while (!eof || tail < head) {
        if (!eof && head - tail < (uint32_t)kSlots) {
            Slot& s = pl.slot[head % kSlots];
            // the host reads chunk `head` while the GPU works on the chunks before it
            const long long got = read(s.h_in, pl.chunk);
            if (got < 0) return fail(ctx, CSVB200_ERR_IO, "input reader reported an error");
            if ((size_t)got < pl.chunk) eof = true;
            if (got > 0 || head == 0) {
                s.bytes = (size_t)got;
                if (s.bytes == 0) {
                    // empty input: the index is the sentinel alone
                    const uint64_t zero = 0;
                    if (direct_dst) {
                        if (direct_cap < 1) dst_small = true;
                        else direct_dst[0] = 0;
                        pl.next_slot_global = 1;
                    } else {
                        if (sink(&zero, 1, 0) != 0) return fail(ctx, CSVB200_ERR_IO, "index sink reported an error");
                        pl.next_slot_global = 1;
                    }
                    break;
                }
                rc = pl.launch(s);
                if (rc) return rc;
                ++head;
            }
            if (head - tail < (uint32_t)kSlots && !eof) continue;   // keep the ring full before blocking on a drain
        }
        if (tail < head) {
            rc = pl.drain(pl.slot[tail % kSlots], sink, direct_dst, direct_cap, &dst_small);
            if (rc) return rc;
            ++tail;
        }
    }
    CU_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (stats) {
        stats->bytes = pl.total_bytes;
        stats->entries = pl.next_slot_global;
        stats->end_parity = pl.end_parity;
        stats->chunks = pl.chunks;
        stats->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    }
    if (dst_small) return fail(ctx, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    return CSVB200_OK;
}

}  // namespace

extern "C" {

int csvb200_index_build_stream(csvb200_ctx* ctx, csvb200_read_fn read_fn, void* read_user, csvb200_sink_fn sink_fn,
                               void* sink_user, size_t chunk_bytes, csvb200_stream_stats* stats)
{
    if (!ctx || !read_fn || !sink_fn) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    // the reader may return short counts before the end of the input: keep asking until the chunk is full
    ReadFn read = [&](uint8_t* dst, size_t cap) -> long long {
        size_t got = 0;
        while (got < cap) {
            const size_t k = read_fn(read_user, dst + got, cap - got);
            if (k == 0) break;
            if (k > cap - got) return -1;
            got += k;
        }
        return (long long)got;
    };
    SinkFn sink = [&](const uint64_t* e, size_t n, uint64_t first) { return sink_fn(sink_user, e, n, first); };
    return run_pipeline(ctx, chunk_bytes, read, sink, nullptr, 0, stats);
}

int csvb200_index_build_file(csvb200_ctx* ctx, const char* path, uint64_t* dst, size_t dst_cap, size_t* len_out,
                             csvb200_stream_stats* stats)
{
    if (!ctx || !path || !len_out || (!dst && dst_cap)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    const int fd = ::open(path, O_RDONLY);
    if (fd < 0) return fail(ctx, CSVB200_ERR_IO, std::string("open ") + path + ": " + std::strerror(errno));   // StructureError::Io
    SlicePool& pool = io_pool(ctx);
    uint64_t file_off = 0;
    bool io_error = false;
    ReadFn read = [&](uint8_t* buf, size_t cap) -> long long {
        // every pool thread preads its own slice of the chunk straight into the pinned buffer
        std::atomic<size_t> total{0};
        pool.run([&](int i, int n) {
            const size_t per = ((cap + n - 1) / n + 4095) & ~size_t(4095);
            size_t a = std::min(cap, per * i);
            const size_t b = std::min(cap, per * (i + 1));
            while (a < b) {
                const ssize_t k = ::pread(fd, buf + a, b - a, (off_t)(file_off + a));
                if (k < 0) {
                    io_error = true;
                    return;
                }
                if (k == 0) break;   // end of file inside (or before) this slice
                a += (size_t)k;
                total += (size_t)k;
            }
        });
        if (io_error) return -1;
        file_off += total.load();
        return (long long)total.load();
    };
    csvb200_stream_stats local{};
    csvb200_stream_stats* st = stats ? stats : &local;
    int rc;
    if (dst && is_pinned(dst)) {
        SinkFn none = [](const uint64_t*, size_t, uint64_t) { return 0; };
        rc = run_pipeline(ctx, 0, read, none, dst, dst_cap, st);
    } else {
        bool small = false;
        SinkFn sink = [&](const uint64_t* e, size_t n, uint64_t first) {
            if (first + n > dst_cap) {
                small = true;        // keep counting so *len_out tells the caller what to allocate
                return 0;
            }
            parallel_memcpy(pool, dst + first, e, n * sizeof(uint64_t));
            return 0;
        };
        rc = run_pipeline(ctx, 0, read, sink, nullptr, 0, st);
        if (!rc && small) rc = fail(ctx, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    }
    ::close(fd);
    *len_out = (size_t)st->entries;
    return rc;
}

}  // extern "C"
