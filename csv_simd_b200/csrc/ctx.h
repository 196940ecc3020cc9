// ctx.h -- private definitions shared by the host-side translation units of libcsvb200
// (api.cu: the C ABI; stream.cu: streaming ingest).  Not part of the public interface.
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../include/csvb200.h"
#include "internal.h"

namespace csvb200 {
class SlicePool;
}

namespace csvb200 {
constexpr size_t kCells = 4096;              // result cells (4 x u64 each): a ring of kRingCells + one scratch cell
constexpr size_t kCellWords = 4;
constexpr size_t kRingCells = kCells - 1;    // the last cell is the out-of-bounds flag of the async seek calls
constexpr uint64_t kDefaultPredictWindow = 64u << 10;
constexpr size_t kStageBytes = 32u << 20;    // pinned staging buffers for pageable input
constexpr int kStageBufs = 2;
constexpr size_t kE2eChunk = 64u << 20;      // H2D / kernel / D2H pipeline granularity
constexpr size_t kBounceEntries = 4u << 20;  // 32 MiB per bounce buffer
}  // namespace csvb200

struct csvb200_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // D2H of finished index segments (overlaps H2D)
    cudaStream_t stream = nullptr;       // the stream work is issued on
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;
    bool timed = false;
    uint8_t* d_scratch = nullptr;  // generic scratch (materialisation): zeroed by its users
    size_t scratch_bytes = 0;
    // scratch of the index builds: [128 B head: ticket, done counter, totals][tagged look-back descriptors]; zeroed when
    // it is (re)allocated and when the 20-bit tag wraps, never between launches
    uint8_t* d_bscratch = nullptr;
    size_t bscratch_bytes = 0;
    uint32_t desc_tag = 0;
    uint64_t* d_cells = nullptr;
    uint64_t* h_cells = nullptr;
    // ownership of the result cells: every live index object, shard job and running pipeline holds its cells
    // until it is freed, so a lazily synced index can never read a cell that was handed to another operation
    std::vector<uint8_t> cell_busy;   // [kRingCells]
    size_t cell_hint = 0;
    // pinned rings of the streaming ingest (stream.cu), kept across calls: page-locking 240 MiB costs ~0.1 s
    uint8_t* h_stream_in[3] = {nullptr, nullptr, nullptr};
    uint64_t* h_stream_out[3] = {nullptr, nullptr, nullptr};
    size_t stream_chunk = 0, stream_out_cap = 0;
    uint64_t* h_bounce[2] = {nullptr, nullptr};   // pinned bounce buffers for index segments headed to pageable memory
    cudaEvent_t bounce_done[2] = {nullptr, nullptr};
    csvb200::SlicePool* pool = nullptr;   // host threads for pread / staging copies, created on first use (io_pool)
    csvb200::SlicePool* pool_down = nullptr;   // a second set for the download side of the pageable pipeline (io_pool_down)
    uint8_t* h_small_in = nullptr;             // pinned, device-mapped staging of the small-input fast path (build_to_host_small)
    uint64_t* h_small_out = nullptr;
    bool dbg_timeline = false;                 // CSVB200_DBG_TIMELINE: device-resident builds run the instrumented kernel
    uint64_t* d_dbg = nullptr;                 // ... and leave 8 words per super-tile here
    size_t dbg_words = 0;
    int io_threads = 0;                        // slices per pool; 0 = default_io_threads() (csvb200_multi_create divides them over its devices)
    uint8_t* h_seek_stage = nullptr;   // pinned staging of the batched seeks from pageable arrays (kept across calls)
    size_t seek_stage_bytes = 0;
    uint8_t* h_stage[csvb200::kStageBufs] = {nullptr, nullptr};
    cudaEvent_t stage_free[csvb200::kStageBufs] = {nullptr, nullptr};
    uint32_t reserve_num = 1, reserve_den = 3;
    // entries per input byte seen by the builds of this context (x 1.25): once known, large builds reserve by it
    // instead of by the 1/3 worst-case guess (a 4 GiB shard reserved 11.5 GB for a 1.9 GB index, and mapping a block of
    // that size for the first time stalls a launch by ~0.3 s); an index that outgrows its reserve is rebuilt exactly
    double density_hint = 0.0;
    bool reserve_explicit = false;    // csvb200_ctx_set_reserve was called: the ratio is the caller's, no hint
    uint64_t launches = 0;
    int kernel_override = 0;  // 0 = auto, 1 = simple, 2 = tma (CSVB200_KERNEL)
    uint32_t tune = 0;        // CSVB200_TUNE: bit 0x400 = the no-chain timing experiment (launch_build)
    const uint8_t* dbg_desc_src = nullptr;   // (debug) input the look-back descriptors in d_bscratch belong to
    size_t dbg_desc_n = 0;
    std::string err;
};

// cross-GPU exchange endpoint of one context (exchange.cu; protocol in internal.h ExchangeArgs)
struct csvb200_exchange {
    csvb200_ctx* ctx = nullptr;
    uint32_t rank = 0, world = 1;
    uint64_t epoch = 0;                                  // builds issued through this endpoint (collective order)
    uint64_t* d_mbox = nullptr;                          // this rank's mailbox (cudaMalloc: IPC-exportable)
    uint64_t* peer[csvb200::kExMaxWorld] = {};           // every rank's mailbox as mapped into this device
    bool ipc_opened[csvb200::kExMaxWorld] = {};
    uint64_t** d_peers = nullptr;                        // device copy of peer[]
    bool connected = false;
    uint64_t timeout_ns = 5000000000ull;                 // CSVB200_EXCHANGE_TIMEOUT_MS (default 5 s)
    uint64_t* d_row4 = nullptr;                          // {entries, end parity, carry used, total} of an end-to-end build
    uint64_t* h_rows = nullptr;                          // pinned: one mailbox slot (host-side wait for all ranks)
};

struct csvb200_index {
    csvb200_ctx* ctx = nullptr;
    uint64_t* d_index = nullptr;
    size_t cap = 0;
    size_t len = 0;
    int end_parity = 0;
    bool synced = false;
    size_t cell = 0;
    cudaEvent_t done = nullptr;
    // inputs of the build, kept for the transparent rebuild on capacity overflow
    const uint8_t* src = nullptr;
    size_t n = 0;
    uint32_t carry_parity = 0;
    uint64_t pos_bias = 0;
    uint64_t out_base = 1;
    const uint32_t* d_shard_par = nullptr;  // device-resident shard parities (multi-GPU), or null
    uint32_t shard_rank = 0;
    uint64_t* d_result2 = nullptr;          // optional caller-owned device copy of {count, parity}
    // speculative sharded build: carry cell {0, carry parity, decisive quote found, redo flag} (device / pinned mirror)
    bool speculative = false;
    bool verified = false;
    // CSVB200_BUILD_VALIDATE: by-products of the build launch
    bool validate = false;
    uint32_t* d_nonascii = nullptr;         // one bit per look-back tile of flag_tile_bytes input bytes
    uint64_t flag_tile_bytes = 0;
    int any_nonascii = 0;
    uint64_t newlines = 0;                  // CR / LF bytes outside quotes
    bool redone_sticky = false;             // the misprediction re-index ran (survives a later capacity rebuild)
    csvb200_exchange* ex = nullptr;         // built with the exchange inside the launch (csvb200_index_build_shard_exchange)
    uint64_t ex_epoch = 0;
    size_t carry_cell = SIZE_MAX;
    uint64_t predict_window = 0;
    uint8_t* d_bytes_owned = nullptr;
    bool borrowed = false;                  // d_index belongs to the caller (csvb200_index_wrap_device): never freed here
    // Tape metadata (TapeCore::init)
    bool tape_ready = false;
    uint32_t field_cnt = 0, record_cnt = 0;
    uint64_t jump = 0;
    int crlf = 0;
};

namespace csvb200 {

int fail(csvb200_ctx* ctx, int code, const std::string& msg);
// `count` consecutive free result cells (first-fit from a rotating hint); SIZE_MAX when the context holds
// kRingCells live cells already
size_t cell_alloc(csvb200_ctx* ctx, size_t count);
void cell_release(csvb200_ctx* ctx, size_t first, size_t count);
// cells held for the duration of one synchronous call
struct CellLease {
    csvb200_ctx* ctx;
    size_t first, count;
    CellLease(csvb200_ctx* c, size_t n) : ctx(c), first(cell_alloc(c, n)), count(n) {}
    CellLease(const CellLease&) = delete;
    CellLease& operator=(const CellLease&) = delete;
    ~CellLease()
    {
        if (ok()) cell_release(ctx, first, count);
    }
    bool ok() const { return first != SIZE_MAX; }
};
int ensure_scratch(csvb200_ctx* ctx, size_t bytes);
// One launch of the index build on `stream`.  The caller fills the input, the output and its capacity, the carry, the
// sentinel and the validate / exchange / speculative extras of p; this fills the rest (tile count, build scratch and
// descriptor tag, the scratch-head counters of the extras, the result cell `cell`), picks the kernel and launches it.
// allow_tma = false: the input is mapped host memory, which only the one-tile-per-CTA kernel reads.
int launch_build(csvb200_ctx* ctx, BuildParams& p, size_t cell, cudaStream_t stream, bool allow_tma = true);
bool is_pinned(const void* p);
SlicePool& io_pool(csvb200_ctx* ctx);   // the context's host-thread pool (CSVB200_IO_THREADS)
// host -> device copy of n bytes on the context's stream; pinned sources go straight to cudaMemcpyAsync,
// pageable ones through the context's pinned staging ring
int upload(csvb200_ctx* ctx, uint8_t* d_dst, const uint8_t* h_src, size_t n);

// cudaMallocAsync from the device's default pool.  The pool keeps every freed block (release threshold = max, set at
// context creation) and, once csvb200_multi_create has granted peer devices access to it, can answer a small request
// with "out of memory" while the device is all but empty (seen on a 2-GPU box: 34 MB refused with 181 GB free, after
// earlier contexts of the process had left cached blocks behind).  Handing the unused blocks back to the driver and
// asking again resolves it, so every stream-ordered allocation of the library goes through here.
inline cudaError_t pool_malloc(void** p, size_t bytes, cudaStream_t s)
{
    cudaError_t e = cudaMallocAsync(p, bytes, s);
    if (e != cudaErrorMemoryAllocation) return e;
    cudaGetLastError();
    int dev = 0;
    cudaMemPool_t pool;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess ||
        cudaDeviceGetDefaultMemPool(&pool, dev) != cudaSuccess) {
        cudaGetLastError();
        return cudaErrorMemoryAllocation;
    }
    cudaMemPoolTrimTo(pool, 0);
    return cudaMallocAsync(p, bytes, s);
}

// stream-ordered device allocation released on scope exit (error paths included)
struct DevBuf {
    void* p = nullptr;
    cudaStream_t stream = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { reset(); }
    cudaError_t alloc(size_t bytes, cudaStream_t s)
    {
        reset();
        stream = s;
        return pool_malloc(&p, bytes ? bytes : 1, s);
    }
    void reset()
    {
        if (p) cudaFreeAsync(p, stream);
        p = nullptr;
    }
    void* release()
    {
        void* r = p;
        p = nullptr;
        return r;
    }
    template <class T>
    T* as() const { return static_cast<T*>(p); }
};

// device -> host copy of `count` index entries on the context's stream, synchronous; a pinned destination is DMA'd in
// place, a pageable one goes through the context's two pinned bounce buffers and its host threads
int download(csvb200_ctx* ctx, uint64_t* dst, const uint64_t* d_src, size_t count);
int ensure_bounce(csvb200_ctx* ctx);
// What the materialisation launches read: the index addressed by global slot (index[s] for s < index_len), the bytes
// the positions point into (bytes[0] is global byte pos_bias, n of them) and the tape metadata.
struct MatSource {
    const uint64_t* index;
    uint64_t index_len;
    const uint8_t* bytes;
    uint64_t n, pos_bias;
    uint32_t record_cnt, field_cnt, row_size;
};
// Enqueues the offsets pass (lengths + scan into d_offsets, offset_base[c] added to column c's; offset_base may be null)
// and / or the write pass of `ncols` columns on the context's stream; one column goes to the single-column kernels.
int materialize_multi_enqueue(csvb200_ctx* ctx, const MatSource& src, const uint32_t* fields, uint32_t ncols,
                              uint32_t first_record, uint32_t nrec, uint32_t flags, uint64_t* const* d_offsets,
                              uint8_t* const* d_outs, const size_t* out_caps, const uint64_t* offset_base, bool offsets_pass,
                              bool write_pass);
// host-side wait for all ranks' rows of one build (exchange.cu)
int exchange_wait_all(csvb200_exchange* ex, uint64_t epoch, uint64_t* counts, uint32_t* carries);

#define CU_TRY(ctx, expr)                                                                       \
    do {                                                                                        \
        cudaError_t e_ = (expr);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            cudaGetLastError();                                                                 \
            return csvb200::fail((ctx), e_ == cudaErrorMemoryAllocation ? CSVB200_ERR_OOM : CSVB200_ERR_CUDA, \
                                 std::string(#expr) + ": " + cudaGetErrorString(e_));           \
        }                                                                                       \
    } while (0)

}  // namespace csvb200
