// api.cu -- the C ABI of libcsvb200 (see include/csvb200.h): context, streams, pinned
// staging, index objects, Tape metadata and lookup entry points.  Host orchestration only;
// all compute is in the kernels (index_build_tma.cu, index_build.cu, lookup.cu, tape.cu, materialize.cu,
// validate.cu); stream.cu holds the streaming-ingest half of the ABI.  There is deliberately no CPU fallback:
// every compute entry point returns CSVB200_ERR_CUDA when the device path is unavailable.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <new>
#include <string>
#include <vector>

#include "ctx.h"
#include "slice_pool.h"

using namespace csvb200;

namespace csvb200 {

int fail(csvb200_ctx* ctx, int code, const std::string& msg)
{
    if (ctx) ctx->err = msg;
    return code;
}

SlicePool& io_pool(csvb200_ctx* ctx)
{
    if (!ctx->pool) ctx->pool = new SlicePool(ctx->io_threads > 0 ? ctx->io_threads : default_io_threads());
    return *ctx->pool;
}

// The pageable end-to-end pipeline copies into staging (uploads) and out of the bounce buffers (downloads) at the
// same time, from two host threads: each side has its own slices (SlicePool::run is one job at a time).
SlicePool& io_pool_down(csvb200_ctx* ctx)
{
    if (!ctx->pool_down) ctx->pool_down = new SlicePool(ctx->io_threads > 0 ? ctx->io_threads : default_io_threads());
    return *ctx->pool_down;
}

bool is_pinned(const void* p)
{
    cudaPointerAttributes attr{};
    const bool ok = cudaPointerGetAttributes(&attr, p) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    return ok;
}

size_t cell_alloc(csvb200_ctx* ctx, size_t count)
{
    if (ctx->cell_busy.empty()) ctx->cell_busy.assign(kRingCells, 0);
    if (count == 0 || count > kRingCells) return SIZE_MAX;
    std::vector<uint8_t>& busy = ctx->cell_busy;
    size_t start = ctx->cell_hint + count <= kRingCells ? ctx->cell_hint : 0;
    for (int pass = 0; pass < 2; ++pass) {
        size_t run = 0;
        for (size_t i = start; i < kRingCells; ++i) {
            run = busy[i] ? 0 : run + 1;
            if (run == count) {
                const size_t first = i + 1 - count;
                std::fill(busy.begin() + first, busy.begin() + i + 1, (uint8_t)1);
                ctx->cell_hint = i + 1 < kRingCells ? i + 1 : 0;
                return first;
            }
        }
        start = 0;
    }
    return SIZE_MAX;
}

void cell_release(csvb200_ctx* ctx, size_t first, size_t count)
{
    if (first == SIZE_MAX || first + count > ctx->cell_busy.size()) return;
    std::fill(ctx->cell_busy.begin() + first, ctx->cell_busy.begin() + first + count, (uint8_t)0);
}

int ensure_scratch(csvb200_ctx* ctx, size_t bytes)
{
    if (bytes <= ctx->scratch_bytes) return CSVB200_OK;
    size_t nb = std::max(bytes, ctx->scratch_bytes * 2);
    nb = (nb + 4095) & ~size_t(4095);
    if (ctx->d_scratch) CU_TRY(ctx, cudaFreeAsync(ctx->d_scratch, ctx->stream));
    ctx->d_scratch = nullptr;
    ctx->scratch_bytes = 0;
    CU_TRY(ctx, pool_malloc((void**)&ctx->d_scratch, nb, ctx->stream));
    ctx->scratch_bytes = nb;
    return CSVB200_OK;
}

// build scratch of at least `bytes` + a fresh descriptor tag for one launch on `stream`
static int next_build_scratch(csvb200_ctx* ctx, size_t bytes, cudaStream_t stream, uint32_t* tag_out, bool reuse_tag)
{
    if (bytes > ctx->bscratch_bytes) {
        size_t nb = std::max(bytes, ctx->bscratch_bytes * 2);
        nb = (nb + 4095) & ~size_t(4095);
        if (ctx->d_bscratch) CU_TRY(ctx, cudaFreeAsync(ctx->d_bscratch, stream));
        ctx->d_bscratch = nullptr;
        ctx->bscratch_bytes = 0;
        CU_TRY(ctx, pool_malloc((void**)&ctx->d_bscratch, nb, stream));
        ctx->bscratch_bytes = nb;
        CU_TRY(ctx, cudaMemsetAsync(ctx->d_bscratch, 0, nb, stream));
        ctx->desc_tag = 0;
    }
    if (!reuse_tag || ctx->desc_tag == 0) {
        if (ctx->desc_tag >= (uint32_t)kTagMask) {   // the tag wraps after a million launches: one full wipe
            CU_TRY(ctx, cudaMemsetAsync(ctx->d_bscratch, 0, ctx->bscratch_bytes, stream));
            ctx->desc_tag = 0;
        }
        ctx->desc_tag += 1;
    }
    *tag_out = ctx->desc_tag;
    return CSVB200_OK;
}

// kernel choice: the TMA pipeline for anything of size, the one-tile-per-CTA kernel for small inputs;
// CSVB200_KERNEL=simple|tma forces one (tests cross-check the two against each other)
static bool build_uses_tma(const csvb200_ctx* ctx, uint64_t n, bool allow_tma)
{
    if (!allow_tma || ctx->kernel_override == 1) return false;
    if (ctx->kernel_override == 2 && n >= 128) return true;
    return tma_path_usable(n);
}

int launch_build(csvb200_ctx* ctx, BuildParams& p, size_t cell, cudaStream_t stream, bool allow_tma)
{
    // an empty input still runs one (empty) tile: its carry / result live on the device
    const uint64_t num_tiles = std::max<uint64_t>(1, (p.n + kTileBytes - 1) / kTileBytes);
    if (num_tiles > 0xffffffffull) return fail(ctx, CSVB200_ERR_INVALID_ARG, "input too large for one launch");
    // DEBUG (CSVB200_TUNE bit 0x400, timing experiments only): reuse the TAG of the previous build of the same
    // address and size, so every look-back finds a published prefix on its first poll -- the kernel without its chain.
    // The result is exact only when the bytes there are unchanged.
    const bool keep_desc = (ctx->tune & 0x400u) && ctx->dbg_desc_src == p.in && ctx->dbg_desc_n == p.n;
    int rc = next_build_scratch(ctx, 128 + num_tiles * kDescStride * sizeof(uint64_t), stream, &p.desc_tag, keep_desc);
    if (rc) return rc;
    ctx->dbg_desc_src = p.in;
    ctx->dbg_desc_n = p.n;
    // the scratch may have moved just now, so its pointers are handed out here.  Head: [0] ticket, [4] CTAs whose
    // look-back role is over, [8] separator total of the exchange, [16] newlines, [24] non-ASCII flag; all zero at
    // launch, put back to zero by the last CTA that uses them
    uint8_t* head = ctx->d_bscratch;
    p.num_tiles = (uint32_t)num_tiles;
    p.ticket = reinterpret_cast<uint32_t*>(head);
    p.desc = reinterpret_cast<uint64_t*>(head + 128);
    if (p.validate || p.ex.peers) {
        p.ex_done = reinterpret_cast<uint32_t*>(head + 4);
        p.scratch_totals = 1u;
    }
    if (p.ex.peers) p.total_out = reinterpret_cast<unsigned long long*>(head + 8);
    if (p.validate) {
        p.nl_out = reinterpret_cast<unsigned long long*>(head + 16);
        p.hi_out = reinterpret_cast<uint32_t*>(head + 24);
    }
    p.result = ctx->d_cells + cell * kCellWords;
    p.result_host = ctx->h_cells + cell * kCellWords;
    CU_TRY(ctx, build_uses_tma(ctx, p.n, allow_tma) ? launch_index_build_tma(p, stream) : launch_index_build(p, stream));
    ctx->launches += 1;
    return CSVB200_OK;
}

}  // namespace csvb200

namespace {

size_t initial_cap(const csvb200_ctx* ctx, size_t n)
{
    const size_t by_ratio = (size_t)((unsigned __int128)n * ctx->reserve_num / ctx->reserve_den) + 4096;
    if (ctx->reserve_explicit || ctx->density_hint <= 0.0 || n < (size_t(1) << 20)) return by_ratio;
    const size_t by_hint = (size_t)((double)n * ctx->density_hint) + 4096;
    return std::min(by_ratio, std::max(by_hint, n / 64 + 4096));
}

// a finished build of n bytes produced len entries: remember the density for the next reservation
void observe_density(csvb200_ctx* ctx, size_t n, size_t len)
{
    if (n < (size_t(1) << 20)) return;
    const double seen = 1.25 * (double)len / (double)n;
    ctx->density_hint = std::max(seen, 0.9 * ctx->density_hint);
}

// worst-case reservation (one entry per byte) for the duration of a scope: re-index paths that must not overflow
struct ReserveAll {
    csvb200_ctx* ctx;
    uint32_t num, den;
    bool explicit_;
    explicit ReserveAll(csvb200_ctx* c) : ctx(c), num(c->reserve_num), den(c->reserve_den), explicit_(c->reserve_explicit)
    {
        ctx->reserve_num = 1;
        ctx->reserve_den = 1;
        ctx->reserve_explicit = true;
    }
    ~ReserveAll()
    {
        ctx->reserve_num = num;
        ctx->reserve_den = den;
        ctx->reserve_explicit = explicit_;
    }
};

// The storage decision, made here only: a build gets 4-byte entries (a compact index) when it is one piece -- one of the
// two non-shard entry points, so no shard offset, exchange or carry from elsewhere -- of at most 4 GiB, whose largest
// position n - 1 fits in 32 bits, and the context was not created with CSVB200_INDEX_ENTRY_BYTES=8.  The entries are then
// the absolute positions themselves: widening one is a zero-extension.  Every other index holds u64 entries.
uint32_t entry_bytes_for(const csvb200_ctx* ctx, size_t n, bool one_piece)
{
    return one_piece && ctx->compact_index && (uint64_t)n <= (1ull << 32) ? 4u : 8u;
}

// enqueue one build of idx->src[0..n) into idx->d_entries (capacity idx->cap)
// redo = the conditional second launch of a speculative shard build (runs only if the carry prediction was wrong)
int enqueue_build(csvb200_index* idx, bool timed, bool redo = false)
{
    csvb200_ctx* ctx = idx->ctx;
    const size_t n = idx->n;
    const uint64_t num_tiles = (n + kTileBytes - 1) / kTileBytes;
    // an empty shard still runs one (empty) tile when its carry / result live on the device
    if (num_tiles == 0 && !(idx->d_shard_par || idx->d_result2 || idx->speculative)) {
        if (idx->out_base == 1 && idx->cap > 0) CU_TRY(ctx, cudaMemsetAsync(idx->d_entries, 0, idx->entry_bytes, ctx->stream));  // sentinel alone
        uint64_t* h_cell = ctx->h_cells + idx->cell * kCellWords;
        h_cell[0] = 0;
        h_cell[1] = idx->carry_parity;
    } else {
        BuildParams p{};
        p.in = idx->src;
        p.n = n;
        p.index = idx->d_entries;
        p.entry_bytes = idx->entry_bytes;
        p.cap = idx->cap;
        p.out_base = idx->out_base;
        p.pos_bias = idx->pos_bias;
        p.carry_parity = idx->carry_parity;
        p.write_sentinel = idx->out_base == 1 ? 1u : 0u;
        p.result2 = idx->d_result2;
        p.result2_words = 2;
        p.shard_par = idx->d_shard_par;
        p.shard_rank = idx->shard_rank;
        if (ctx->dbg_timeline && !redo && !idx->validate && !idx->ex) {   // debug: per-super-tile timestamps of this build
            const size_t words = 8 * (num_tiles + 1);
            if (ctx->dbg_words < words) {
                if (ctx->d_dbg) cudaFree(ctx->d_dbg);
                ctx->d_dbg = nullptr;
                ctx->dbg_words = 0;
                if (cudaMalloc((void**)&ctx->d_dbg, words * sizeof(uint64_t)) == cudaSuccess) ctx->dbg_words = words;
            }
            if (ctx->d_dbg) {
                CU_TRY(ctx, cudaMemsetAsync(ctx->d_dbg, 0, ctx->dbg_words * sizeof(uint64_t), ctx->stream));
                p.dbg = ctx->d_dbg;
            }
        }
        const bool use_tma = build_uses_tma(ctx, n, true);
        if (idx->validate) {
            // by-products: newline count and non-ASCII flag accumulate in the zeroed head of the scratch, the per-tile
            // non-ASCII bitmap belongs to the index (K7 later visits the flagged tiles only)
            const size_t words = (size_t)(num_tiles + 31) / 32;
            if (!idx->d_nonascii) CU_TRY(ctx, pool_malloc((void**)&idx->d_nonascii, words * sizeof(uint32_t), ctx->stream));
            CU_TRY(ctx, cudaMemsetAsync(idx->d_nonascii, 0, words * sizeof(uint32_t), ctx->stream));
            idx->flag_tile_bytes = build_flag_tile_bytes(use_tma);
            p.validate = 1u;
            p.nonascii_bitmap = idx->d_nonascii;
        }
        if (idx->speculative) {
            uint64_t* d_carry = ctx->d_cells + idx->carry_cell * kCellWords;
            p.carry = d_carry;
            p.result2_words = 4;
            if (redo) {
                p.run_flag = reinterpret_cast<const uint32_t*>(d_carry + 3);
            } else if (idx->ex) {
                // exchange inside the launch: separator total and the "look-back role over" counter live in the
                // zeroed head of the scratch; the last CTA posts the row and resolves the carry chain into d_carry
                p.ex.peers = idx->ex->d_peers;
                p.ex.rank = idx->ex->rank;
                p.ex.world = idx->ex->world;
                p.ex.epoch = idx->ex_epoch;
                p.ex.timeout_ns = idx->ex->timeout_ns;
                p.ex.out = d_carry;
                p.ex.out_host = ctx->h_cells + idx->carry_cell * kCellWords;
            } else if (!idx->verified && idx->d_result2) {
                // first (speculative) launch: also accumulate the shard's separator total
                CU_TRY(ctx, cudaMemsetAsync(idx->d_result2, 0, 4 * sizeof(uint64_t), ctx->stream));
                p.total_out = reinterpret_cast<unsigned long long*>(idx->d_result2 + 3);
            }
        }
        // the conditional re-index of the exchange form sits right behind the build: launched programmatically
        // dependent, its CTAs are scheduled as the build's CTAs leave, wait for the build's completion inside the kernel and
        // exit on the flag -- the launch latency hides behind the build's tail
        if (redo && idx->ex && use_tma) p.pdl_wait = 2u;
        if (timed) CU_TRY(ctx, cudaEventRecord(ctx->ev_k0, ctx->stream));
        if (idx->speculative && !redo && !idx->verified) {
            // predicted carry-in parity (rank 0 and empty shards: known to be 0) into the device cell the launch reads;
            // the predictor sits right in front of the build so that the build can start under it (pdl_wait)
            uint64_t* d_carry = ctx->d_cells + idx->carry_cell * kCellWords;
            if (idx->shard_rank == 0 || n == 0) {
                CU_TRY(ctx, cudaMemsetAsync(d_carry, 0, kCellWords * sizeof(uint64_t), ctx->stream));
            } else {
                CU_TRY(ctx, launch_predict_carry(idx->src, n, idx->predict_window, d_carry, ctx->stream));
                ctx->launches += 1;
                p.pdl_wait = use_tma ? 1u : 0u;
            }
        }
        const int rc = launch_build(ctx, p, idx->cell, ctx->stream);
        if (rc) return rc;
        if (timed) {
            CU_TRY(ctx, cudaEventRecord(ctx->ev_k1, ctx->stream));
            ctx->timed = true;
        }
    }
    CU_TRY(ctx, cudaEventRecord(idx->done, ctx->stream));
    idx->synced = false;
    return CSVB200_OK;
}

int new_index(csvb200_ctx* ctx, csvb200_index** out)
{
    csvb200_index* idx = new (std::nothrow) csvb200_index();
    if (!idx) return fail(ctx, CSVB200_ERR_OOM, "host allocation failed");
    idx->ctx = ctx;
    idx->cell = cell_alloc(ctx, 1);
    if (idx->cell == SIZE_MAX) {
        delete idx;
        return fail(ctx, CSVB200_ERR_OOM, "too many live index objects in this context (4095 result cells)");
    }
    cudaError_t e = cudaEventCreateWithFlags(&idx->done, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        cell_release(ctx, idx->cell, 1);
        delete idx;
        return fail(ctx, CSVB200_ERR_CUDA, std::string("cudaEventCreate: ") + cudaGetErrorString(e));
    }
    *out = idx;
    return CSVB200_OK;
}

int build_device_common(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t carry_parity, uint64_t pos_bias,
                        int emit_sentinel, csvb200_index** out, const uint32_t* d_shard_par = nullptr,
                        uint32_t shard_rank = 0, uint64_t* d_result2 = nullptr, bool speculative = false,
                        uint64_t predict_window = 0, csvb200_exchange* ex = nullptr, bool validate = false,
                        bool one_piece = false)
{
    if (!ctx || !out || (n && !dev_bytes)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    if ((reinterpret_cast<uintptr_t>(dev_bytes) & 15u) != 0)
        return fail(ctx, CSVB200_ERR_INVALID_ARG, "device input must be 16-byte aligned");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    csvb200_index* idx = nullptr;
    int rc = new_index(ctx, &idx);
    if (rc) return rc;
    idx->src = static_cast<const uint8_t*>(dev_bytes);
    idx->n = n;
    idx->carry_parity = carry_parity & 1u;
    idx->pos_bias = pos_bias;
    idx->out_base = emit_sentinel ? 1 : 0;
    idx->d_shard_par = d_shard_par;
    idx->shard_rank = shard_rank;
    idx->d_result2 = d_result2;
    idx->validate = validate;
    if (ex) {
        idx->ex = ex;
        idx->ex_epoch = ++ex->epoch;
    }
    if (speculative) {
        // predicted carry-in parity (rank 0: known to be 0) in a device cell the build launch reads
        idx->carry_cell = cell_alloc(ctx, 1);
        if (idx->carry_cell == SIZE_MAX) {
            csvb200_index_free(idx);
            return fail(ctx, CSVB200_ERR_OOM, "too many live index objects in this context (4095 result cells)");
        }
        idx->speculative = true;
        idx->predict_window = predict_window ? predict_window : kDefaultPredictWindow;
    }
    idx->entry_bytes = entry_bytes_for(ctx, n, one_piece && pos_bias == 0 && !ex && !speculative && !d_shard_par && !d_result2);
    idx->cap = initial_cap(ctx, n);
    const size_t idx_bytes = idx->cap * idx->entry_bytes;
    cudaError_t e = pool_malloc(&idx->d_entries, idx_bytes, ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        csvb200_index_free(idx);
        size_t mem_free = 0, mem_total = 0;
        cudaMemGetInfo(&mem_free, &mem_total);
        cudaGetLastError();
        return fail(ctx, CSVB200_ERR_OOM, "index allocation of " + std::to_string(idx_bytes) + " bytes on device " +
                                              std::to_string(ctx->device) + ": " + cudaGetErrorString(e) + " (" +
                                              std::to_string(mem_free >> 20) + " of " + std::to_string(mem_total >> 20) + " MiB free)");
    }
    rc = enqueue_build(idx, true);
    if (!rc && ex) {
        // the rebuild with the true carry is enqueued unconditionally and exits at once when the flag is 0
        idx->verified = true;
        rc = enqueue_build(idx, false, true);
    }
    if (rc) {
        csvb200_index_free(idx);
        return rc;
    }
    *out = idx;
    return CSVB200_OK;
}

}  // namespace

namespace csvb200 {

// host -> device copy of n bytes; pinned sources go straight to cudaMemcpyAsync, pageable ones
// through the context's pinned staging ring.
int upload(csvb200_ctx* ctx, uint8_t* d_dst, const uint8_t* h_src, size_t n)
{
    if (n == 0) return CSVB200_OK;
    if (is_pinned(h_src)) {
        CU_TRY(ctx, cudaMemcpyAsync(d_dst, h_src, n, cudaMemcpyHostToDevice, ctx->stream));
        return CSVB200_OK;
    }
    for (int b = 0; b < kStageBufs; ++b) {
        if (!ctx->h_stage[b]) {
            CU_TRY(ctx, cudaHostAlloc((void**)&ctx->h_stage[b], kStageBytes, cudaHostAllocDefault));
            CU_TRY(ctx, cudaEventCreateWithFlags(&ctx->stage_free[b], cudaEventDisableTiming));
        }
    }
    size_t off = 0;
    int b = 0;
    while (off < n) {
        const size_t len = std::min(kStageBytes, n - off);
        CU_TRY(ctx, cudaEventSynchronize(ctx->stage_free[b]));
        parallel_memcpy(io_pool(ctx), ctx->h_stage[b], h_src + off, len, CopyDir::ToStaging);   // one thread cannot feed PCIe
        CU_TRY(ctx, cudaMemcpyAsync(d_dst + off, ctx->h_stage[b], len, cudaMemcpyHostToDevice, ctx->stream));
        CU_TRY(ctx, cudaEventRecord(ctx->stage_free[b], ctx->stream));
        off += len;
        b = (b + 1) % kStageBufs;
    }
    return CSVB200_OK;
}

int ensure_bounce(csvb200_ctx* ctx)
{
    for (int i = 0; i < 2; ++i) {
        cudaError_t e = cudaSuccess;
        if (!ctx->h_bounce[i]) e = cudaHostAlloc((void**)&ctx->h_bounce[i], kBounceEntries * sizeof(uint64_t), cudaHostAllocDefault);
        if (e == cudaSuccess && !ctx->bounce_done[i]) e = cudaEventCreateWithFlags(&ctx->bounce_done[i], cudaEventDisableTiming);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, CSVB200_ERR_OOM, std::string("bounce buffers: ") + cudaGetErrorString(e));
        }
    }
    return CSVB200_OK;
}

int download(csvb200_ctx* ctx, uint64_t* dst, const uint64_t* d_src, size_t count)
{
    if (count == 0) return CSVB200_OK;
    if (!dst || !d_src) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (is_pinned(dst)) {
        CU_TRY(ctx, cudaMemcpyAsync(dst, d_src, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        return CSVB200_OK;
    }
    int rc = ensure_bounce(ctx);
    if (rc) return rc;
    size_t pos[2] = {0, 0}, len[2] = {0, 0}, issued = 0, flushed = 0;
    auto flush = [&](size_t k) -> cudaError_t {
        const int b = (int)(k & 1);
        cudaError_t e = cudaEventSynchronize(ctx->bounce_done[b]);
        if (e == cudaSuccess) parallel_memcpy(io_pool(ctx), dst + pos[b], ctx->h_bounce[b], len[b] * sizeof(uint64_t));
        return e;
    };
    for (size_t off = 0; off < count; off += kBounceEntries) {
        const int b = (int)(issued & 1);
        if (issued >= 2) CU_TRY(ctx, flush(flushed++));
        pos[b] = off;
        len[b] = std::min(kBounceEntries, count - off);
        CU_TRY(ctx, cudaMemcpyAsync(ctx->h_bounce[b], d_src + off, len[b] * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(ctx, cudaEventRecord(ctx->bounce_done[b], ctx->stream));
        ++issued;
    }
    while (flushed < issued) CU_TRY(ctx, flush(flushed++));
    return CSVB200_OK;
}

}  // namespace csvb200

extern "C" {

int csvb200_version(void) { return CSVB200_VERSION; }

const char* csvb200_status_string(int s)
{
    switch (s) {
    case CSVB200_OK: return "ok";
    case CSVB200_ERR_INVALID_ARG: return "invalid argument";
    case CSVB200_ERR_INVALID_STATE: return "Invalid state";
    case CSVB200_ERR_INVALID_CSV_FORMAT: return "Unsupported csv structure: likely variable number of fields";
    case CSVB200_ERR_MISSING_VALUE: return "Missing a value";
    case CSVB200_ERR_IO: return "io error";
    case CSVB200_ERR_CUDA: return "CUDA error";
    case CSVB200_ERR_OOM: return "out of memory";
    case CSVB200_ERR_INPUT_TOO_SMALL: return "input shorter than 64 bytes";
    case CSVB200_ERR_CAPACITY: return "destination capacity too small";
    case CSVB200_ERR_OUT_OF_BOUNDS: return "index slot out of bounds";
    case CSVB200_ERR_EXCHANGE: return "cross-GPU exchange failed";
    default: return "unknown status";
    }
}

int csvb200_ctx_create(int device, csvb200_ctx** out)
{
    if (!out) return CSVB200_ERR_INVALID_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
        cudaGetLastError();
        return CSVB200_ERR_CUDA;  // no CPU fallback by design
    }
    csvb200_ctx* ctx = new (std::nothrow) csvb200_ctx();
    if (!ctx) return CSVB200_ERR_OOM;
    ctx->device = device;
    if (const char* k = std::getenv("CSVB200_KERNEL")) {
        if (std::strcmp(k, "simple") == 0) ctx->kernel_override = 1;
        if (std::strcmp(k, "tma") == 0) ctx->kernel_override = 2;
    }
    if (const char* t = std::getenv("CSVB200_TUNE")) ctx->tune = (uint32_t)std::atoi(t);
    ctx->dbg_timeline = std::getenv("CSVB200_DBG_TIMELINE") != nullptr;
    if (const char* b = std::getenv("CSVB200_INDEX_ENTRY_BYTES")) ctx->compact_index = std::strcmp(b, "8") != 0;
    auto bail = [&](cudaError_t) {
        cudaGetLastError();
        csvb200_ctx_destroy(ctx);
        return (int)CSVB200_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail(e);
    if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    if ((e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(e);
    ctx->stream = ctx->own_stream;
    if ((e = cudaEventCreate(&ctx->ev_k0)) != cudaSuccess) return bail(e);
    if ((e = cudaEventCreate(&ctx->ev_k1)) != cudaSuccess) return bail(e);
    if ((e = cudaMalloc((void**)&ctx->d_cells, kCells * kCellWords * sizeof(uint64_t))) != cudaSuccess) return bail(e);
    if ((e = cudaHostAlloc((void**)&ctx->h_cells, kCells * kCellWords * sizeof(uint64_t), cudaHostAllocMapped | cudaHostAllocPortable)) !=
        cudaSuccess)
        return bail(e);
    // keep freed blocks in the stream-ordered pool so per-build allocations are reused, not re-mapped
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        uint64_t thr = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    cudaGetLastError();
    *out = ctx;
    return CSVB200_OK;
}

void csvb200_ctx_destroy(csvb200_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->own_stream) cudaStreamSynchronize(ctx->own_stream);
    if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
    if (ctx->d_scratch) cudaFree(ctx->d_scratch);
    if (ctx->d_bscratch) cudaFree(ctx->d_bscratch);
    if (ctx->d_cells) cudaFree(ctx->d_cells);
    if (ctx->h_cells) cudaFreeHost(ctx->h_cells);
    delete ctx->pool;
    delete ctx->pool_down;
    if (ctx->d_dbg) cudaFree(ctx->d_dbg);
    if (ctx->h_small_in) cudaFreeHost(ctx->h_small_in);
    if (ctx->h_small_out) cudaFreeHost(ctx->h_small_out);
    for (int i = 0; i < 2; ++i) {
        if (ctx->h_bounce[i]) cudaFreeHost(ctx->h_bounce[i]);
        if (ctx->bounce_done[i]) cudaEventDestroy(ctx->bounce_done[i]);
    }
    if (ctx->h_seek_stage) cudaFreeHost(ctx->h_seek_stage);
    for (int i = 0; i < 3; ++i) {
        if (ctx->h_stream_in[i]) cudaFreeHost(ctx->h_stream_in[i]);
        if (ctx->h_stream_out[i]) cudaFreeHost(ctx->h_stream_out[i]);
    }
    for (int b = 0; b < kStageBufs; ++b) {
        if (ctx->h_stage[b]) cudaFreeHost(ctx->h_stage[b]);
        if (ctx->stage_free[b]) cudaEventDestroy(ctx->stage_free[b]);
    }
    if (ctx->ev_k0) cudaEventDestroy(ctx->ev_k0);
    if (ctx->ev_k1) cudaEventDestroy(ctx->ev_k1);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    cudaGetLastError();
    delete ctx;
}

const char* csvb200_last_error(const csvb200_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int csvb200_ctx_set_stream(csvb200_ctx* ctx, void* cuda_stream)
{
    if (!ctx) return CSVB200_ERR_INVALID_ARG;
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->own_stream;
    return CSVB200_OK;
}

int csvb200_ctx_set_reserve(csvb200_ctx* ctx, uint32_t num, uint32_t den)
{
    if (!ctx || den == 0) return fail(ctx, CSVB200_ERR_INVALID_ARG, "bad reserve ratio");
    ctx->reserve_num = num;
    ctx->reserve_den = den;
    ctx->reserve_explicit = true;
    return CSVB200_OK;
}

int csvb200_ctx_last_build_ms(csvb200_ctx* ctx, float* ms)
{
    if (!ctx || !ms) return CSVB200_ERR_INVALID_ARG;
    if (!ctx->timed) return fail(ctx, CSVB200_ERR_INVALID_STATE, "no timed build yet");
    CU_TRY(ctx, cudaEventSynchronize(ctx->ev_k1));
    CU_TRY(ctx, cudaEventElapsedTime(ms, ctx->ev_k0, ctx->ev_k1));
    return CSVB200_OK;
}

uint64_t csvb200_ctx_launch_count(const csvb200_ctx* ctx) { return ctx ? ctx->launches : 0; }

int csvb200_host_alloc(size_t bytes, void** out)
{
    if (!out) return CSVB200_ERR_INVALID_ARG;
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? CSVB200_ERR_OOM : CSVB200_ERR_CUDA;
    }
    return CSVB200_OK;
}

int csvb200_host_free(void* p)
{
    if (!p) return CSVB200_OK;
    return cudaFreeHost(p) == cudaSuccess ? CSVB200_OK : CSVB200_ERR_CUDA;
}

// Debug export (not part of include/csvb200.h): the timeline words of the last build made under CSVB200_DBG_TIMELINE.
int csvb200_debug_timeline(csvb200_ctx* ctx, uint64_t* dst, size_t cap_words, size_t* words)
{
    if (!ctx || !words) return CSVB200_ERR_INVALID_ARG;
    *words = ctx->dbg_words;
    if (!dst || cap_words < ctx->dbg_words || !ctx->d_dbg) return ctx->d_dbg ? CSVB200_ERR_CAPACITY : CSVB200_ERR_INVALID_STATE;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    CU_TRY(ctx, cudaMemcpy(dst, ctx->d_dbg, ctx->dbg_words * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return CSVB200_OK;
}

int csvb200_host_register(void* p, size_t bytes, int read_only)
{
    if (!p || bytes == 0) return CSVB200_ERR_INVALID_ARG;
    cudaError_t e = cudaHostRegister(p, bytes, read_only ? cudaHostRegisterReadOnly : cudaHostRegisterDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        if (e == cudaErrorMemoryAllocation) return CSVB200_ERR_OOM;
        return (e == cudaErrorHostMemoryAlreadyRegistered || e == cudaErrorInvalidValue || e == cudaErrorNotSupported)
                   ? CSVB200_ERR_INVALID_ARG
                   : CSVB200_ERR_CUDA;
    }
    return CSVB200_OK;
}

int csvb200_host_unregister(void* p)
{
    if (!p) return CSVB200_ERR_INVALID_ARG;
    cudaError_t e = cudaHostUnregister(p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return e == cudaErrorHostMemoryNotRegistered || e == cudaErrorInvalidValue ? CSVB200_ERR_INVALID_ARG : CSVB200_ERR_CUDA;
    }
    return CSVB200_OK;
}

int csvb200_index_build_device(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t flags, csvb200_index** out)
{
    if (ctx && (flags & CSVB200_BUILD_STRICT_MIN64) && n < 64)
        return fail(ctx, CSVB200_ERR_INPUT_TOO_SMALL, "n < 64: the reference panics on this input");
    return build_device_common(ctx, dev_bytes, n, 0u, 0ull, 1, out, nullptr, 0, nullptr, false, 0, nullptr,
                               (flags & CSVB200_BUILD_VALIDATE) != 0, true);
}

int csvb200_index_validation(csvb200_index* idx, int* is_ascii, uint64_t* newlines_outside_quotes)
{
    if (!idx) return CSVB200_ERR_INVALID_ARG;
    if (!idx->validate) return fail(idx->ctx, CSVB200_ERR_INVALID_STATE, "index was built without CSVB200_BUILD_VALIDATE");
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    if (is_ascii) *is_ascii = idx->any_nonascii ? 0 : 1;
    if (newlines_outside_quotes) *newlines_outside_quotes = idx->newlines;
    return CSVB200_OK;
}

int csvb200_index_validate_utf8(csvb200_index* idx, uint64_t* valid_up_to)
{
    if (!idx || !valid_up_to) return CSVB200_ERR_INVALID_ARG;
    if (!idx->validate) return fail(idx->ctx, CSVB200_ERR_INVALID_STATE, "index was built without CSVB200_BUILD_VALIDATE");
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    csvb200_ctx* ctx = idx->ctx;
    *valid_up_to = UINT64_MAX;
    if (!idx->any_nonascii || idx->n == 0) return CSVB200_OK;   // ASCII is well-formed UTF-8: nothing to read again
    const uint8_t* bytes = idx->d_bytes_owned ? idx->d_bytes_owned : idx->src;
    if (!bytes) return fail(ctx, CSVB200_ERR_INVALID_STATE, "index was built without CSVB200_BUILD_KEEP_BYTES");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CellLease lease(ctx, 1);
    if (!lease.ok()) return fail(ctx, CSVB200_ERR_OOM, "no free result cell (4095 live index objects)");
    uint64_t* d_cell = ctx->d_cells + lease.first * kCellWords;
    uint64_t* h_cell = ctx->h_cells + lease.first * kCellWords;
    CU_TRY(ctx, cudaMemsetAsync(d_cell, 0xff, sizeof(uint64_t), ctx->stream));
    CU_TRY(ctx, launch_utf8_validate_flagged(bytes, idx->n, idx->d_nonascii, idx->flag_tile_bytes, d_cell, ctx->stream));
    ctx->launches += 1;
    CU_TRY(ctx, cudaMemcpyAsync(h_cell, d_cell, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *valid_up_to = h_cell[0];
    return CSVB200_OK;
}

int csvb200_index_build_shard_device(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t carry_parity,
                                     uint64_t global_offset, int emit_sentinel, csvb200_index** out)
{
    return build_device_common(ctx, dev_bytes, n, carry_parity, global_offset, emit_sentinel, out);
}

int csvb200_index_build_shard_device_ex(csvb200_ctx* ctx, const void* dev_bytes, size_t n,
                                        const uint32_t* d_shard_parities, uint32_t shard_rank, uint64_t global_offset,
                                        int emit_sentinel, uint64_t* d_result_out, csvb200_index** out)
{
    if (ctx && !d_shard_parities) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null shard parity array");
    return build_device_common(ctx, dev_bytes, n, 0u, global_offset, emit_sentinel, out, d_shard_parities, shard_rank,
                               d_result_out);
}

int csvb200_index_build_shard_speculative(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t shard_rank,
                                          uint64_t global_offset, int emit_sentinel, uint64_t predict_window,
                                          uint64_t* d_result_out, csvb200_index** out)
{
    if (ctx && !d_result_out) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null result array");
    return build_device_common(ctx, dev_bytes, n, 0u, global_offset, emit_sentinel, out, nullptr, shard_rank, d_result_out,
                               true, predict_window);
}

int csvb200_index_build_shard_exchange(csvb200_ctx* ctx, csvb200_exchange* ex, const void* dev_bytes, size_t n,
                                       uint64_t global_offset, uint64_t predict_window, csvb200_index** out)
{
    if (!ctx || !ex || ex->ctx != ctx) return fail(ctx, CSVB200_ERR_INVALID_ARG, "exchange does not belong to this context");
    if (!ex->connected) return fail(ctx, CSVB200_ERR_INVALID_STATE, "exchange is not connected");
    return build_device_common(ctx, dev_bytes, n, 0u, global_offset, ex->rank == 0 ? 1 : 0, out, nullptr, ex->rank, nullptr,
                               true, predict_window, ex);
}

int csvb200_index_shard_info(csvb200_index* idx, csvb200_shard_info* out)
{
    if (!idx || !out) return CSVB200_ERR_INVALID_ARG;
    if (!idx->ex) return fail(idx->ctx, CSVB200_ERR_INVALID_STATE, "index was not built through an exchange");
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    const uint64_t* h_carry = idx->ctx->h_cells + idx->carry_cell * kCellWords;
    const uint64_t below = h_carry[2] & ~(1ull << 63);
    out->entries = idx->len;
    out->base = idx->ex->rank == 0 ? 0 : 1 + below;
    out->carry_in = (uint32_t)(h_carry[1] & 1u);
    out->redone = idx->redone_sticky ? 1u : 0u;
    out->rank = idx->ex->rank;
    out->world = idx->ex->world;
    out->epoch = idx->ex_epoch;
    return CSVB200_OK;
}

int csvb200_index_shard_verify(csvb200_index* idx, const uint64_t* d_gathered, uint32_t world, uint64_t* d_final_out)
{
    if (!idx) return CSVB200_ERR_INVALID_ARG;
    csvb200_ctx* ctx = idx->ctx;
    if (!idx->speculative) return fail(ctx, CSVB200_ERR_INVALID_STATE, "index was not built speculatively");
    if (!d_gathered || idx->shard_rank >= world) return fail(ctx, CSVB200_ERR_INVALID_ARG, "bad gathered array / world size");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    uint64_t* d_carry = ctx->d_cells + idx->carry_cell * kCellWords;
    uint64_t* h_carry = ctx->h_cells + idx->carry_cell * kCellWords;
    CU_TRY(ctx, launch_verify_carry(d_gathered, world, idx->shard_rank, d_carry, d_final_out, ctx->stream));
    ctx->launches += 1;
    idx->verified = true;
    CU_TRY(ctx, cudaMemcpyAsync(h_carry, d_carry, kCellWords * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    // the rebuild with the true carry is enqueued unconditionally and exits at once when the flag is 0
    return enqueue_build(idx, false, true);
}

int csvb200_index_shard_redone(csvb200_index* idx, int* redone, int* carry_parity)
{
    if (!idx) return CSVB200_ERR_INVALID_ARG;
    if (!idx->speculative || !idx->verified)
        return fail(idx->ctx, CSVB200_ERR_INVALID_STATE, "csvb200_index_shard_verify has not been called");
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    const uint64_t* h_carry = idx->ctx->h_cells + idx->carry_cell * kCellWords;
    if (redone) *redone = idx->redone_sticky ? 1 : 0;
    if (carry_parity) *carry_parity = (int)(h_carry[1] & 1u);
    return CSVB200_OK;
}

int csvb200_shard_quote_parity_device(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t* d_parity_out)
{
    if (!ctx || !d_parity_out || (n && !dev_bytes)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    if ((reinterpret_cast<uintptr_t>(dev_bytes) & 15u) != 0)
        return fail(ctx, CSVB200_ERR_INVALID_ARG, "device input must be 16-byte aligned");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaMemsetAsync(d_parity_out, 0, sizeof(uint32_t), ctx->stream));
    CU_TRY(ctx, launch_quote_parity(static_cast<const uint8_t*>(dev_bytes), n, d_parity_out, ctx->stream));
    if (n) ctx->launches += 1;
    return CSVB200_OK;
}

int csvb200_index_build(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint32_t flags, csvb200_index** out)
{
    if (!ctx || !out || (n && !host_bytes)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    if ((flags & CSVB200_BUILD_STRICT_MIN64) && n < 64)
        return fail(ctx, CSVB200_ERR_INPUT_TOO_SMALL, "n < 64: the reference panics on this input");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    DevBuf d_bytes;
    CU_TRY(ctx, d_bytes.alloc(((n + 15) & ~size_t(15)) + 16, ctx->stream));
    int rc = upload(ctx, d_bytes.as<uint8_t>(), host_bytes, n);
    csvb200_index* idx = nullptr;
    if (!rc) rc = build_device_common(ctx, d_bytes.p, n, 0u, 0ull, 1, &idx, nullptr, 0, nullptr, false, 0, nullptr,
                                      (flags & CSVB200_BUILD_VALIDATE) != 0, true);
    if (!rc) rc = csvb200_index_sync(idx);  // resolves a capacity overflow while the bytes are still here
    if (rc) {
        if (idx) csvb200_index_free(idx);
        return rc;
    }
    if (flags & CSVB200_BUILD_KEEP_BYTES)
        idx->d_bytes_owned = static_cast<uint8_t*>(d_bytes.release());
    else
        idx->src = nullptr;   // d_bytes is released (stream-ordered) on return
    *out = idx;
    return CSVB200_OK;
}

// Simple (non-overlapped) form: build on the device, then copy the index out.
static int build_to_host_serial(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* dst, size_t dst_cap,
                                size_t* len_out)
{
    csvb200_index* idx = nullptr;
    int rc = csvb200_index_build(ctx, host_bytes, n, CSVB200_BUILD_DEFAULT, &idx);
    if (rc) return rc;
    *len_out = idx->len;
    rc = idx->len <= dst_cap ? csvb200_index_copy_out(idx, dst, dst_cap)
                             : fail(ctx, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    csvb200_index_free(idx);
    return rc;
}

// Small inputs (<= 256 KiB): the call is all latency -- two copies, a stream-ordered allocation, two synchronisations
// around a ~5 us kernel cost 46-63 us, while the reference's loop indexes 64 KiB in 10 us.  Here the kernel reads the
// bytes straight out of pinned host memory and writes the entries straight into pinned host memory (zero-copy over
// PCIe; both buffers are the context's own and reused, or the caller's destination when that is pinned): one launch, one
// synchronisation, no device allocation.
constexpr size_t kSmallDirectBytes = 256u << 10;
static int build_to_host_small(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* dst, size_t dst_cap,
                               size_t* len_out)
{
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    if (!ctx->h_small_in) {
        CU_TRY(ctx, cudaHostAlloc((void**)&ctx->h_small_in, kSmallDirectBytes + 64, cudaHostAllocMapped));
        CU_TRY(ctx, cudaHostAlloc((void**)&ctx->h_small_out, (kSmallDirectBytes + 2) * sizeof(uint64_t), cudaHostAllocMapped));
    }
    std::memcpy(ctx->h_small_in, host_bytes, n);
    bool direct = is_pinned(dst) && (reinterpret_cast<uintptr_t>(dst) & 7u) == 0;
    void* dst_dev = nullptr;
    if (direct && (cudaHostGetDevicePointer(&dst_dev, dst, 0) != cudaSuccess || dst_dev != static_cast<void*>(dst))) {
        cudaGetLastError();
        direct = false;   // pinned, but not addressable from the device under the same pointer: stage it
    }
    uint64_t* out = direct ? dst : ctx->h_small_out;
    const size_t cap = direct ? dst_cap : kSmallDirectBytes + 2;
    CellLease lease(ctx, 1);
    if (!lease.ok()) return fail(ctx, CSVB200_ERR_OOM, "no free result cell (4095 live index objects)");
    BuildParams p{};
    p.in = ctx->h_small_in;       // unified addressing: pinned host memory is addressable from the device as it is
    p.n = n;
    p.index = out;
    p.cap = cap;
    p.out_base = 1;
    p.write_sentinel = 1u;
    int rc = launch_build(ctx, p, lease.first, ctx->stream, false);
    if (rc) return rc;
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    const size_t len = 1 + (size_t)ctx->h_cells[lease.first * kCellWords];
    *len_out = len;
    if (len > dst_cap) return fail(ctx, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    if (!direct) std::memcpy(dst, ctx->h_small_out, len * sizeof(uint64_t));
    return CSVB200_OK;
}

// End-to-end pipeline: the input goes up in kE2eChunk pieces, each piece is indexed by its own launch
// chained to the previous one through a device-resident carry cell {entries so far, quote parity}
// (no host round trip between launches), and every finished index segment goes down on a second
// stream while later pieces are still going up -- PCIe is full duplex, so the step costs about
// max(H2D, D2H) instead of their sum.
namespace {
struct PipeOpts {
    uint64_t pos_bias = 0;           // global byte offset of host_bytes[0] (shards)
    int emit_sentinel = 1;
    bool predict = false;            // shard, first attempt: guess the carry-in parity from the bytes of chunk 0
    const uint64_t* d_carry0 = nullptr;   // shard, second attempt: device cell {0, true carry parity}
    uint64_t* d_result4 = nullptr;   // optional device words {entries excl. sentinel, end parity, carry used, separator total}
    const uint8_t* d_bytes_in = nullptr;  // the bytes are already on the device (rebuild): no uploads
    uint8_t** keep_bytes = nullptr;  // receives the device copy of the input instead of freeing it
};

// overflow_out: the index reserve was too small (the caller decides how to rebuild); dst_small_out (optional):
// the caller's array was too small (*len_out says how many entries there are) -- an error when it is null
int pipeline_to_host(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* dst, size_t dst_cap, size_t* len_out,
                     const PipeOpts& o, bool* overflow_out, bool* dst_small_out = nullptr)
{
    // chunk schedule: the downloads cannot start before the first chunk is up and indexed, so the pipeline ramps
    // up (chunk/8, chunk/4, chunk/2, then full chunks) instead of paying a full chunk of upload time as fill latency
    // (measured: 27.16 vs 27.28 ms per GiB of cfg2 -- the step is bound by the D2H volume, the fill is ~1 ms of it)
    std::vector<size_t> chunk_off;
    {
        static_assert(kE2eChunk / 8 % 128 == 0, "chunk boundaries stay 128-byte aligned (TMA rows)");
        size_t off = 0, len = kE2eChunk / 8;
        while (off < n) {
            chunk_off.push_back(off);
            off += std::min(len, n - off);
            len = std::min(kE2eChunk, len * 2);
        }
        if (chunk_off.empty()) chunk_off.push_back(0);   // an empty shard still runs one empty launch
        chunk_off.push_back(n);
    }
    const size_t nchunks = chunk_off.size() - 1;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    // cells: cell0 = carry into chunk 0; cell[c+1] = result of chunk c (held until this call returns)
    CellLease lease(ctx, nchunks + 1);
    if (!lease.ok()) return fail(ctx, CSVB200_ERR_OOM, "not enough free result cells for the chunk pipeline");
    const size_t cell0 = lease.first;
    cudaStream_t s_up = ctx->stream, s_down = ctx->copy_stream;
    uint8_t* d_bytes = const_cast<uint8_t*>(o.d_bytes_in);
    uint64_t* d_index = nullptr;
    const size_t cap = initial_cap(ctx, n);
    const uint64_t out_base = o.emit_sentinel ? 1 : 0;
    if (!d_bytes) CU_TRY(ctx, pool_malloc((void**)&d_bytes, ((n + 15) & ~size_t(15)) + 16, s_up));
    CU_TRY(ctx, pool_malloc((void**)&d_index, cap * sizeof(uint64_t), s_up));
    uint64_t* d_cells = ctx->d_cells + cell0 * kCellWords;
    uint64_t* h_cells = ctx->h_cells + cell0 * kCellWords;
    if (o.d_carry0)
        CU_TRY(ctx, cudaMemcpyAsync(d_cells, o.d_carry0, 2 * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s_up));
    else
        CU_TRY(ctx, cudaMemsetAsync(d_cells, 0, kCellWords * sizeof(uint64_t), s_up));
    if (o.d_result4) CU_TRY(ctx, cudaMemsetAsync(o.d_result4, 0, 4 * sizeof(uint64_t), s_up));
    std::vector<cudaEvent_t> done(nchunks, nullptr);
    int rc = CSVB200_OK;
    auto cleanup = [&]() {
        for (cudaEvent_t e : done)
            if (e) cudaEventDestroy(e);
        cudaStreamSynchronize(s_down);
        if (o.keep_bytes && rc == CSVB200_OK)
            *o.keep_bytes = d_bytes;
        else if (!o.d_bytes_in)
            cudaFreeAsync(d_bytes, s_up);
        cudaFreeAsync(d_index, s_up);
    };
    // ---- enqueue every upload + launch ----
    // Pinned (or device-resident) input: nothing here waits on the host, the whole schedule is enqueued before the first
    // download is looked at.  Pageable input: every upload is a host copy into pinned staging, so this side runs on its
    // own thread and the calling thread starts the downloads as the chunks finish -- the two host copies (input into
    // staging, index out of the bounce buffers) and the two DMA directions all overlap.
    std::atomic<size_t> enqueued{0};       // chunks whose `done` event is recorded
    std::atomic<bool> enqueue_failed{false};
    int rc_up = CSVB200_OK;
    auto enqueue_all = [&]() {
      int& rc = rc_up;
      if (cudaSetDevice(ctx->device) != cudaSuccess) rc = CSVB200_ERR_CUDA;
      for (size_t c = 0; c < nchunks && rc == CSVB200_OK; ++c) {
        const size_t off = chunk_off[c], len = chunk_off[c + 1] - off;
        if (!o.d_bytes_in) rc = upload(ctx, d_bytes + off, host_bytes + off, len);
        if (rc) break;
        cudaError_t e = cudaSuccess;
        if (c == 0 && o.predict && len > 0) {
            e = launch_predict_carry(d_bytes, len, kDefaultPredictWindow, d_cells, s_up);   // cell0 <- {0, guess, found, 0}
            ctx->launches += 1;
        }
        BuildParams p{};
        p.in = d_bytes + off;
        p.n = len;                         // an empty shard runs one empty tile
        p.index = d_index;
        p.cap = cap;
        p.out_base = out_base;
        p.pos_bias = o.pos_bias + off;
        p.carry = d_cells + c * kCellWords;
        p.write_sentinel = (c == 0 && out_base) ? 1u : 0u;
        if (o.d_result4) p.total_out = reinterpret_cast<unsigned long long*>(o.d_result4 + 3);
        if (e == cudaSuccess) {
            rc = launch_build(ctx, p, cell0 + c + 1, s_up);
            if (rc) break;
            e = cudaEventCreateWithFlags(&done[c], cudaEventDisableTiming);
        }
        if (e == cudaSuccess) e = cudaEventRecord(done[c], s_up);
        if (e != cudaSuccess) {
            cudaGetLastError();
            rc = fail(ctx, CSVB200_ERR_CUDA, std::string("e2e pipeline: ") + cudaGetErrorString(e));
        }
        if (rc == CSVB200_OK) enqueued.store(c + 1, std::memory_order_release);
      }
      if (rc == CSVB200_OK && o.d_result4) {
          // {entries, end parity} of the last chunk, the carry parity the first chunk used; the separator total was
          // accumulated by the launches themselves
          cudaError_t e = cudaMemcpyAsync(o.d_result4, d_cells + nchunks * kCellWords, 2 * sizeof(uint64_t), cudaMemcpyDeviceToDevice, s_up);
          if (e == cudaSuccess) e = cudaMemcpyAsync(o.d_result4 + 2, d_cells + 1, sizeof(uint64_t), cudaMemcpyDeviceToDevice, s_up);
          if (e != cudaSuccess) {
              cudaGetLastError();
              rc = fail(ctx, CSVB200_ERR_CUDA, std::string("e2e pipeline: ") + cudaGetErrorString(e));
          }
      }
      if (rc != CSVB200_OK) enqueue_failed.store(true, std::memory_order_release);
    };
    const bool two_threads = !o.d_bytes_in && n >= (64u << 20) && !is_pinned(host_bytes);
    std::thread uploader;
    bool spawned = false;
    if (two_threads) {
        try {
            uploader = std::thread(enqueue_all);
            spawned = true;
        } catch (...) {   // no thread to be had: enqueue on this one, as for pinned input
        }
    }
    if (!spawned) {
        enqueue_all();
        rc = rc_up;
    }
    // ---- as each chunk's kernel finishes, send its index segment down on the second stream ----
    // A pinned destination is DMA'd in place.  A pageable one (a plain Vec<usize>) would make every copy a
    // synchronous driver-staged transfer, so its segments come down into two pinned bounce buffers and the
    // context's host threads move them on while the next piece is in flight.
    const bool bounce = dst != nullptr && !is_pinned(dst);
    if (bounce && rc == CSVB200_OK) rc = ensure_bounce(ctx);
    size_t piece_pos[2] = {0, 0}, piece_len[2] = {0, 0}, pieces = 0, flushed = 0;
    auto flush_piece = [&](size_t k) -> cudaError_t {   // piece k (in order): wait for its D2H, copy it to dst
        const int b = (int)(k & 1);
        cudaError_t e = cudaEventSynchronize(ctx->bounce_done[b]);
        if (e == cudaSuccess) parallel_memcpy(io_pool_down(ctx), dst + piece_pos[b], ctx->h_bounce[b], piece_len[b] * sizeof(uint64_t));
        return e;
    };
    size_t copied = 0;  // entries already on their way to dst (including the sentinel)
    bool overflow = false, dst_small = false;
    for (size_t c = 0; c < nchunks && rc == CSVB200_OK; ++c) {
        while (enqueued.load(std::memory_order_acquire) <= c && !enqueue_failed.load(std::memory_order_acquire))
            std::this_thread::yield();     // (pageable input) the uploader has not reached this chunk yet
        if (enqueued.load(std::memory_order_acquire) <= c) break;   // the uploader failed: its status is reported below
        cudaError_t e = cudaEventSynchronize(done[c]);
        if (e == cudaSuccess) {
            const size_t upto = (size_t)out_base + (size_t)h_cells[(c + 1) * kCellWords];  // entries through this chunk
            if (upto > cap) overflow = true;
            if (upto > dst_cap || (upto && !dst)) dst_small = true;
            if (!overflow && !dst_small && upto > copied) {
                e = cudaStreamWaitEvent(s_down, done[c], 0);
                if (!bounce) {
                    if (e == cudaSuccess)
                        e = cudaMemcpyAsync(dst + copied, d_index + copied, (upto - copied) * sizeof(uint64_t),
                                            cudaMemcpyDeviceToHost, s_down);
                } else {
                    for (size_t pos = copied; pos < upto && e == cudaSuccess; pos += kBounceEntries) {
                        const size_t len = std::min(kBounceEntries, upto - pos);
                        const int b = (int)(pieces & 1);
                        if (pieces >= 2) {   // the buffer still holds piece (pieces - 2): move it on first
                            e = flush_piece(flushed++);
                            if (e != cudaSuccess) break;
                        }
                        e = cudaMemcpyAsync(ctx->h_bounce[b], d_index + pos, len * sizeof(uint64_t), cudaMemcpyDeviceToHost, s_down);
                        if (e == cudaSuccess) e = cudaEventRecord(ctx->bounce_done[b], s_down);
                        piece_pos[b] = pos;
                        piece_len[b] = len;
                        ++pieces;
                    }
                }
                copied = upto;
            }
            if (c + 1 == nchunks) {
                *len_out = upto;
                observe_density(ctx, n, upto);
            }
        }
        if (e != cudaSuccess) {
            cudaGetLastError();
            rc = fail(ctx, CSVB200_ERR_CUDA, std::string("e2e pipeline: ") + cudaGetErrorString(e));
        }
    }
    while (rc == CSVB200_OK && flushed < pieces) {
        if (flush_piece(flushed++) != cudaSuccess) {
            cudaGetLastError();
            rc = fail(ctx, CSVB200_ERR_CUDA, "e2e pipeline: bounce copy failed");
        }
    }
    if (uploader.joinable()) uploader.join();
    if (rc == CSVB200_OK) rc = rc_up;
    if (rc == CSVB200_OK) {
        cudaError_t e = cudaStreamSynchronize(s_down);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s_up);
        if (e != cudaSuccess) rc = fail(ctx, CSVB200_ERR_CUDA, std::string("e2e pipeline: ") + cudaGetErrorString(e));
    }
    cleanup();
    if (rc) return rc;
    *overflow_out = overflow;
    if (dst_small_out) *dst_small_out = dst_small;
    if (!overflow && dst_small && !dst_small_out) return fail(ctx, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    return CSVB200_OK;
}
}  // namespace

int csvb200_index_build_to_host(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* dst, size_t dst_cap,
                                size_t* len_out)
{
    if (!ctx || !len_out || (n && !host_bytes)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    // (CSVB200_KERNEL=tma sends small inputs to the general path: the zero-copy one runs the one-tile-per-CTA kernel only)
    if (n > 0 && n <= kSmallDirectBytes && dst && ctx->kernel_override != 2) return build_to_host_small(ctx, host_bytes, n, dst, dst_cap, len_out);
    const size_t nchunks = (n + kE2eChunk - 1) / kE2eChunk;
    if (nchunks < 2 || nchunks + 1 >= kRingCells || !dst) return build_to_host_serial(ctx, host_bytes, n, dst, dst_cap, len_out);
    bool overflow = false;
    int rc = pipeline_to_host(ctx, host_bytes, n, dst, dst_cap, len_out, PipeOpts{}, &overflow);
    if (rc) return rc;
    if (overflow) return build_to_host_serial(ctx, host_bytes, n, dst, dst_cap, len_out);  // denser than the reserve
    return CSVB200_OK;
}

// ---- end-to-end form of the speculative sharded build --------------------------------------------------------
struct csvb200_shard_job {
    csvb200_ctx* ctx = nullptr;
    const uint8_t* host_bytes = nullptr;
    size_t n = 0;
    uint32_t rank = 0;
    uint64_t global_offset = 0;
    int emit_sentinel = 0;
    uint64_t* dst = nullptr;
    size_t dst_cap = 0;
    uint64_t* d_result4 = nullptr;
    uint8_t* d_bytes = nullptr;     // device copy of the shard, kept until the job is verified
    size_t carry_cell = 0;
    size_t len = 0;                 // entries in dst after the speculative attempt
    bool dst_small = false;         // ... which did not fit dst (only an error if the guess turns out right)
    bool verified = false;
};

int csvb200_shard_build_to_host(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint32_t shard_rank,
                                uint64_t global_offset, int emit_sentinel, uint64_t* dst, size_t dst_cap, size_t* len_out,
                                uint64_t* d_result_out, csvb200_shard_job** job_out)
{
    if (!ctx || !len_out || !d_result_out || !job_out || (n && !host_bytes)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    csvb200_shard_job* job = new (std::nothrow) csvb200_shard_job();
    if (!job) return fail(ctx, CSVB200_ERR_OOM, "host allocation failed");
    job->ctx = ctx;
    job->host_bytes = host_bytes;
    job->n = n;
    job->rank = shard_rank;
    job->global_offset = global_offset;
    job->emit_sentinel = emit_sentinel;
    job->dst = dst;
    job->dst_cap = dst_cap;
    job->d_result4 = d_result_out;
    job->carry_cell = cell_alloc(ctx, 1);
    if (job->carry_cell == SIZE_MAX) {
        delete job;
        return fail(ctx, CSVB200_ERR_OOM, "too many live objects in this context (4095 result cells)");
    }
    PipeOpts o;
    o.pos_bias = global_offset;
    o.emit_sentinel = emit_sentinel;
    o.predict = shard_rank != 0;          // rank 0 starts outside quotes by definition
    o.d_result4 = d_result_out;
    o.keep_bytes = &job->d_bytes;
    bool overflow = false;
    int rc = pipeline_to_host(ctx, host_bytes, n, dst, dst_cap, len_out, o, &overflow, &job->dst_small);
    if (!rc && overflow) {
        // denser than the reserve: raise the reserve to the worst case for this context and go again
        ReserveAll worst(ctx);
        cudaFreeAsync(job->d_bytes, ctx->stream);
        job->d_bytes = nullptr;
        rc = pipeline_to_host(ctx, host_bytes, n, dst, dst_cap, len_out, o, &overflow, &job->dst_small);
    }
    if (rc) {
        if (job->d_bytes) cudaFreeAsync(job->d_bytes, ctx->stream);
        cell_release(ctx, job->carry_cell, 1);
        delete job;
        return rc;
    }
    job->len = *len_out;
    *job_out = job;
    return CSVB200_OK;
}

int csvb200_shard_job_verify(csvb200_shard_job* job, const uint64_t* d_gathered, uint32_t world, uint64_t* d_final_out,
                             size_t* len_out, int* redone)
{
    if (!job || !d_gathered || !len_out) return CSVB200_ERR_INVALID_ARG;
    csvb200_ctx* ctx = job->ctx;
    if (job->rank >= world) return fail(ctx, CSVB200_ERR_INVALID_ARG, "bad world size");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    uint64_t* d_carry = ctx->d_cells + job->carry_cell * kCellWords;
    uint64_t* h_carry = ctx->h_cells + job->carry_cell * kCellWords;
    CU_TRY(ctx, launch_verify_carry(d_gathered, world, job->rank, d_carry, d_final_out, ctx->stream));
    ctx->launches += 1;
    CU_TRY(ctx, cudaMemcpyAsync(h_carry, d_carry, kCellWords * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    job->verified = true;
    const bool redo = (h_carry[3] & 1u) != 0;
    if (redone) *redone = redo ? 1 : 0;
    *len_out = job->len;
    if (!redo) return job->dst_small ? fail(ctx, CSVB200_ERR_CAPACITY, "destination index buffer too small") : CSVB200_OK;
    // the guess was wrong: index the shard again (it is still on the device) with the true carry
    PipeOpts o;
    o.pos_bias = job->global_offset;
    o.emit_sentinel = job->emit_sentinel;
    o.d_carry0 = d_carry;
    o.d_bytes_in = job->d_bytes;
    o.d_result4 = job->d_result4;
    bool overflow = false;
    ReserveAll worst(ctx);   // a flipped carry can turn every masked separator into an entry
    return pipeline_to_host(ctx, job->host_bytes, job->n, job->dst, job->dst_cap, len_out, o, &overflow);
}

void csvb200_shard_job_free(csvb200_shard_job* job)
{
    if (!job) return;
    cudaSetDevice(job->ctx->device);
    if (job->d_bytes) cudaFreeAsync(job->d_bytes, job->ctx->stream);
    cudaGetLastError();
    cell_release(job->ctx, job->carry_cell, 1);
    delete job;
}

int csvb200_shard_build_to_host_exchange(csvb200_ctx* ctx, csvb200_exchange* ex, const uint8_t* host_bytes, size_t n,
                                         uint64_t global_offset, uint64_t* dst, size_t dst_cap, size_t* len_out,
                                         csvb200_shard_info* info, uint64_t* counts, uint32_t* carries)
{
    if (!ctx || !ex || ex->ctx != ctx || !len_out) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument / foreign exchange");
    if (!ex->connected) return fail(ctx, CSVB200_ERR_INVALID_STATE, "exchange is not connected");
    // 1. the shard goes up, is indexed and comes down chunk by chunk under the predicted carry
    csvb200_shard_job* job = nullptr;
    int rc = csvb200_shard_build_to_host(ctx, host_bytes, n, ex->rank, global_offset, ex->rank == 0 ? 1 : 0, dst, dst_cap, len_out,
                                         ex->d_row4, &job);
    if (rc) return rc;
    // 2. post the row, resolve the lower ranks (one tiny launch; the pipeline's last chunk is not known in advance)
    const uint64_t epoch = ++ex->epoch;
    uint64_t* d_carry = ctx->d_cells + job->carry_cell * kCellWords;
    uint64_t* h_carry = ctx->h_cells + job->carry_cell * kCellWords;
    ExchangeArgs a{};
    a.peers = ex->d_peers;
    a.rank = ex->rank;
    a.world = ex->world;
    a.epoch = epoch;
    a.timeout_ns = ex->timeout_ns;
    a.out = d_carry;
    a.out_host = h_carry;
    cudaError_t e = launch_exchange(a, ex->d_row4, ctx->stream);
    ctx->launches += 1;
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        csvb200_shard_job_free(job);
        return fail(ctx, CSVB200_ERR_CUDA, std::string("exchange launch: ") + cudaGetErrorString(e));
    }
    if (h_carry[2] >> 63) {
        csvb200_shard_job_free(job);
        return fail(ctx, CSVB200_ERR_EXCHANGE, "exchange: a lower rank never posted its row for this build (timeout), or lapped the mailbox ring");
    }
    const bool redo = (h_carry[3] & 1u) != 0;
    // 3. only a shard whose guess was wrong is indexed again, from the device copy the job kept
    if (redo) {
        PipeOpts o;
        o.pos_bias = global_offset;
        o.emit_sentinel = ex->rank == 0 ? 1 : 0;
        o.d_carry0 = d_carry;
        o.d_bytes_in = job->d_bytes;
        bool overflow = false;
        ReserveAll worst(ctx);   // a flipped carry can turn every masked separator into an entry
        rc = pipeline_to_host(ctx, host_bytes, n, dst, dst_cap, len_out, o, &overflow);
    } else if (job->dst_small) {
        rc = fail(ctx, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    }
    if (info) {
        info->entries = *len_out;
        info->base = ex->rank == 0 ? 0 : 1 + (h_carry[2] & ~(1ull << 63));
        info->carry_in = (uint32_t)(h_carry[1] & 1u);
        info->redone = redo ? 1u : 0u;
        info->rank = ex->rank;
        info->world = ex->world;
        info->epoch = epoch;
    }
    csvb200_shard_job_free(job);
    if (!rc && (counts || carries)) rc = exchange_wait_all(ex, epoch, counts, carries);
    return rc;
}

int csvb200_shard_quote_parity(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint32_t* parity_out)
{
    if (!ctx || !parity_out || (n && !dev_bytes)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    if ((reinterpret_cast<uintptr_t>(dev_bytes) & 15u) != 0)
        return fail(ctx, CSVB200_ERR_INVALID_ARG, "device input must be 16-byte aligned");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CellLease lease(ctx, 1);
    if (!lease.ok()) return fail(ctx, CSVB200_ERR_OOM, "no free result cell (4095 live index objects)");
    const size_t cell = lease.first;
    uint64_t* d_cell = ctx->d_cells + cell * kCellWords;
    uint64_t* h_cell = ctx->h_cells + cell * kCellWords;
    CU_TRY(ctx, cudaMemsetAsync(d_cell, 0, sizeof(uint64_t), ctx->stream));
    CU_TRY(ctx, launch_quote_parity(static_cast<const uint8_t*>(dev_bytes), n, reinterpret_cast<uint32_t*>(d_cell),
                                    ctx->stream));
    if (n) ctx->launches += 1;
    CU_TRY(ctx, cudaMemcpyAsync(h_cell, d_cell, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *parity_out = (uint32_t)(h_cell[0] & 1u);
    return CSVB200_OK;
}

int csvb200_index_wrap_device(csvb200_ctx* ctx, const uint64_t* d_entries, size_t len, size_t input_bytes,
                              const void* d_bytes, csvb200_index** out)
{
    if (!ctx || !out || !d_entries || len == 0) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument / empty index");
    if ((reinterpret_cast<uintptr_t>(d_bytes) & 15u) != 0 || (reinterpret_cast<uintptr_t>(d_entries) & 7u) != 0)
        return fail(ctx, CSVB200_ERR_INVALID_ARG, "device input must be 16-byte aligned, entries 8-byte aligned");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    csvb200_index* idx = nullptr;
    int rc = new_index(ctx, &idx);
    if (rc) return rc;
    idx->d_entries = const_cast<uint64_t*>(d_entries);
    idx->borrowed = true;
    idx->cap = idx->len = len;
    idx->n = input_bytes;
    idx->src = static_cast<const uint8_t*>(d_bytes);   // optional: enables tape_validate / materialize / gather
    idx->synced = true;
    *out = idx;
    return CSVB200_OK;
}

int csvb200_index_sync(csvb200_index* idx)
{
    if (!idx) return CSVB200_ERR_INVALID_ARG;
    if (idx->synced) return CSVB200_OK;
    csvb200_ctx* ctx = idx->ctx;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    for (int attempt = 0; attempt < 2; ++attempt) {
        CU_TRY(ctx, cudaEventSynchronize(idx->done));
        const uint64_t* h_cell = ctx->h_cells + idx->cell * kCellWords;
        const size_t len = (size_t)(idx->out_base + h_cell[0]);
        idx->end_parity = (int)(h_cell[1] & 1u);
        if (idx->speculative && idx->verified && (ctx->h_cells[idx->carry_cell * kCellWords + 3] & 1u)) idx->redone_sticky = true;
        if (idx->ex && (ctx->h_cells[idx->carry_cell * kCellWords + 2] >> 63))
            return fail(ctx, CSVB200_ERR_EXCHANGE, "exchange: a lower rank never posted its row for this build (timeout), or lapped the mailbox ring");
        if (len <= idx->cap) {
            idx->len = len;
            observe_density(ctx, idx->n, len);
            if (idx->validate) {
                idx->any_nonascii = idx->n ? (int)(h_cell[2] & 1u) : 0;
                idx->newlines = idx->n ? h_cell[3] : 0;
            }
            idx->synced = true;
            return CSVB200_OK;
        }
        // capacity overflow (denser than the reserve heuristic): rebuild with the exact size
        if (!idx->src) return fail(ctx, CSVB200_ERR_INVALID_STATE, "index overflow and input no longer available");
        CU_TRY(ctx, cudaFreeAsync(idx->d_entries, ctx->stream));
        idx->d_entries = nullptr;
        idx->cap = len + 2;
        CU_TRY(ctx, pool_malloc(&idx->d_entries, idx->cap * idx->entry_bytes, ctx->stream));
        int rc = enqueue_build(idx, true);
        if (rc) return rc;
    }
    return fail(ctx, CSVB200_ERR_CUDA, "index rebuild did not converge");
}

size_t csvb200_index_len(csvb200_index* idx)
{
    if (!idx || csvb200_index_sync(idx) != CSVB200_OK) return 0;
    return idx->len;
}

int csvb200_index_end_parity(csvb200_index* idx)
{
    if (!idx || csvb200_index_sync(idx) != CSVB200_OK) return -1;
    return idx->end_parity;
}

// A compact index turns into an ordinary u64 one, in place and once: whoever asks for raw u64 device memory gets an
// index whose every later consumer takes the u64 path.
static int widen_in_place(csvb200_index* idx)
{
    csvb200_ctx* ctx = idx->ctx;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    DevBuf wide;
    CU_TRY(ctx, wide.alloc(idx->len * sizeof(uint64_t), ctx->stream));
    CU_TRY(ctx, launch_widen_entries(static_cast<const uint32_t*>(idx->d_entries), idx->len, wide.as<uint64_t>(), ctx->stream));
    ctx->launches += 1;
    CU_TRY(ctx, cudaFreeAsync(idx->d_entries, ctx->stream));
    idx->d_entries = wide.release();
    idx->entry_bytes = 8;
    idx->cap = idx->len;
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return CSVB200_OK;
}

const uint64_t* csvb200_index_device_ptr(csvb200_index* idx)
{
    if (!idx || csvb200_index_sync(idx) != CSVB200_OK) return nullptr;
    if (idx->entry_bytes == 4 && widen_in_place(idx) != CSVB200_OK) return nullptr;
    return static_cast<const uint64_t*>(idx->d_entries);
}

constexpr size_t kWidenChunk = 4u << 20;   // entries per widened chunk of a compact index on its way out (32 MiB as u64)

int csvb200_index_copy_out(csvb200_index* idx, uint64_t* dst, size_t dst_cap)
{
    if (!idx || !dst) return CSVB200_ERR_INVALID_ARG;
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    csvb200_ctx* ctx = idx->ctx;
    if (idx->len > dst_cap) return fail(ctx, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    if (idx->entry_bytes == 8) {
        CU_TRY(ctx, cudaMemcpyAsync(dst, idx->d_entries, idx->len * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        return CSVB200_OK;
    }
    // compact index: widened on the device, chunk by chunk, into two pooled buffers; the context's stream widens chunk
    // k + 1 while its copy stream brings chunk k home (widening on the host would cost more than the copy, DESIGN 6)
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t chunk = std::min(kWidenChunk, idx->len);
    DevBuf wide;
    CU_TRY(ctx, wide.alloc(2 * chunk * sizeof(uint64_t), ctx->stream));
    cudaEvent_t widened = nullptr, copied[2] = {nullptr, nullptr};
    cudaError_t e = cudaEventCreateWithFlags(&widened, cudaEventDisableTiming);
    for (int b = 0; b < 2 && e == cudaSuccess; ++b) e = cudaEventCreateWithFlags(&copied[b], cudaEventDisableTiming);
    const uint32_t* src = static_cast<const uint32_t*>(idx->d_entries);
    for (size_t off = 0, k = 0; off < idx->len && e == cudaSuccess; off += chunk, ++k) {
        const size_t len = std::min(chunk, idx->len - off);
        uint64_t* buf = wide.as<uint64_t>() + (k & 1) * chunk;
        if (k >= 2) e = cudaStreamWaitEvent(ctx->stream, copied[k & 1], 0);   // the copy of chunk k - 2 has left buf
        if (e == cudaSuccess) e = launch_widen_entries(src + off, len, buf, ctx->stream);
        if (e == cudaSuccess) ctx->launches += 1;
        if (e == cudaSuccess) e = cudaEventRecord(widened, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, widened, 0);
        if (e == cudaSuccess) e = cudaMemcpyAsync(dst + off, buf, len * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->copy_stream);
        if (e == cudaSuccess) e = cudaEventRecord(copied[k & 1], ctx->copy_stream);
    }
    // the buffers go back to the pool on ctx->stream: it must not run ahead of the last copy
    const cudaError_t s = cudaStreamSynchronize(ctx->copy_stream);
    if (e == cudaSuccess) e = s;
    if (widened) cudaEventDestroy(widened);
    for (cudaEvent_t ev : copied)
        if (ev) cudaEventDestroy(ev);
    CU_TRY(ctx, e);
    return CSVB200_OK;
}

void csvb200_index_free(csvb200_index* idx)
{
    if (!idx) return;
    csvb200_ctx* ctx = idx->ctx;
    cudaSetDevice(ctx->device);
    if (idx->d_entries && !idx->borrowed) cudaFreeAsync(idx->d_entries, ctx->stream);
    if (idx->d_bytes_owned) cudaFreeAsync(idx->d_bytes_owned, ctx->stream);
    if (idx->d_nonascii) cudaFreeAsync(idx->d_nonascii, ctx->stream);
    if (idx->done) cudaEventDestroy(idx->done);
    cudaGetLastError();
    // (a cell released while its launch is still in flight is safe: the next holder's launch follows it in stream order)
    cell_release(ctx, idx->cell, 1);
    if (idx->carry_cell != SIZE_MAX) cell_release(ctx, idx->carry_cell, 1);
    delete idx;
}

int csvb200_tape_init(csvb200_index* idx, uint32_t field_cnt, int crlf, uint32_t* record_cnt, uint64_t* jump)
{
    if (!idx) return CSVB200_ERR_INVALID_ARG;
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    csvb200_ctx* ctx = idx->ctx;
    const uint64_t j = crlf ? (uint64_t)field_cnt + 1 : (uint64_t)field_cnt;  // src/tape.rs:318-321
    if (j == 0 || idx->len == 0) return fail(ctx, CSVB200_ERR_INVALID_ARG, "field_cnt must be >= 1");
    idx->field_cnt = field_cnt;
    idx->crlf = crlf ? 1 : 0;
    idx->jump = j;
    idx->record_cnt = (uint32_t)((idx->len - 1) / j);  // src/tape.rs:323-325
    idx->tape_ready = true;
    if (record_cnt) *record_cnt = idx->record_cnt;
    if (jump) *jump = j;
    if ((idx->len - 1) % j != 0)  // src/tape.rs:327,342-344
        return fail(ctx, CSVB200_ERR_INVALID_CSV_FORMAT, csvb200_status_string(CSVB200_ERR_INVALID_CSV_FORMAT));
    return CSVB200_OK;
}

int csvb200_tape_validate(csvb200_index* idx, uint32_t field_cnt, int crlf, csvb200_tape_report* out)
{
    if (!idx || !out) return CSVB200_ERR_INVALID_ARG;
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    csvb200_ctx* ctx = idx->ctx;
    const uint64_t j = crlf ? (uint64_t)field_cnt + 1 : (uint64_t)field_cnt;  // src/tape.rs:318-321
    if (j == 0 || idx->len == 0) return fail(ctx, CSVB200_ERR_INVALID_ARG, "field_cnt must be >= 1");
    const uint8_t* bytes = idx->d_bytes_owned ? idx->d_bytes_owned : idx->src;
    if (!bytes && idx->n) return fail(ctx, CSVB200_ERR_INVALID_STATE, "index was built without CSVB200_BUILD_KEEP_BYTES");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CellLease lease(ctx, 1);
    if (!lease.ok()) return fail(ctx, CSVB200_ERR_OOM, "no free result cell (4095 live index objects)");
    const size_t cell = lease.first;
    uint64_t* d_cell = ctx->d_cells + cell * kCellWords;
    uint64_t* h_cell = ctx->h_cells + cell * kCellWords;
    CU_TRY(ctx, cudaMemsetAsync(d_cell, 0xff, sizeof(uint64_t), ctx->stream));
    TapeValidateParams p{};
    p.index = idx->d_entries;
    p.entry_bytes = idx->entry_bytes;
    p.index_len = idx->len;
    p.bytes = bytes;
    p.n = idx->n;
    p.pos_bias = idx->pos_bias;
    p.jump = j;
    p.crlf = crlf ? 1 : 0;
    p.first_bad_slot = d_cell;
    CU_TRY(ctx, launch_tape_validate(p, ctx->stream));
    if (idx->len > 1) ctx->launches += 1;
    CU_TRY(ctx, cudaMemcpyAsync(h_cell, d_cell, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    std::memset(out, 0, sizeof(*out));
    out->index_len = idx->len;
    out->jump = j;
    out->record_cnt = (uint32_t)((idx->len - 1) / j);   // src/tape.rs:323-325
    out->problem = (idx->len - 1) % j;                  // src/tape.rs:327
    out->first_bad_slot = h_cell[0];
    out->first_bad_record = UINT64_MAX;
    out->first_bad_pos = UINT64_MAX;
    if (out->first_bad_slot != UINT64_MAX) {
        out->first_bad_record = (out->first_bad_slot - 1) / j;
        out->first_bad_pos = 0;   // a u32 entry lands in the low half (little-endian host)
        CU_TRY(ctx, cudaMemcpyAsync(&out->first_bad_pos,
                                    static_cast<const uint8_t*>(idx->d_entries) + out->first_bad_slot * idx->entry_bytes,
                                    idx->entry_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    } else if (out->problem != 0) {
        out->first_bad_record = (idx->len - 1) / j;      // the file ends inside this record
    }
    out->ok = out->first_bad_slot == UINT64_MAX && out->problem == 0;
    return CSVB200_OK;
}

}  // extern "C"

namespace csvb200 {

int tape_chunk_slots(uint32_t record_cnt, uint64_t jump, uint8_t num, csvb200_chunk* out, size_t out_cap, size_t* n_out)
{
    // boundaries(record_cnt, num) (src/tape.rs:385-428); None -> StructureError::InvalidState (:99-100)
    const uint32_t task = record_cnt;
    if (task == 0 || num == 0) return CSVB200_ERR_INVALID_STATE;
    const size_t nchunks = task < num ? 1 : num;
    *n_out = nchunks;
    if (!out || out_cap < nchunks) return CSVB200_ERR_CAPACITY;
    const uint32_t job = task < num ? task : task / num, rem = task < num ? 0 : task % num;
    uint64_t acc = 0;
    for (size_t i = 0; i < nchunks; ++i) {
        const uint32_t len = job + (i < rem ? 1u : 0u);
        out[i].id = (uint8_t)i;
        out[i].start = acc * jump;                            // KeyToPos(boundary.start * jump) (:104-106)
        out[i].end = (acc + len) * jump;                      // (:107-110)
        out[i].record_cnt = len;
        acc += len;
    }
    out[0].start = jump;                                      // chunk 0 skips the header row (:117-123)
    out[0].record_cnt -= 1;
    return CSVB200_OK;
}

const char* tape_chunk_error(int code)
{
    return code == CSVB200_ERR_CAPACITY ? "chunk array too small" : csvb200_status_string(code);
}

}  // namespace csvb200

extern "C" {

int csvb200_tape_chunks(csvb200_index* idx, uint8_t num, csvb200_chunk* out, size_t out_cap, size_t* n_out)
{
    if (!idx || !n_out) return CSVB200_ERR_INVALID_ARG;
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    csvb200_ctx* ctx = idx->ctx;
    if (!idx->tape_ready) return fail(ctx, CSVB200_ERR_INVALID_STATE, "csvb200_tape_init has not been called");
    rc = tape_chunk_slots(idx->record_cnt, idx->jump, num, out, out_cap, n_out);
    if (rc) return fail(ctx, rc, tape_chunk_error(rc));
    const size_t nchunks = *n_out;
    // byte ranges the chunks delimit: two index entries per chunk, fetched in one small gather
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    std::vector<uint64_t> slots(2 * nchunks), vals(2 * nchunks, UINT64_MAX);
    for (size_t i = 0; i < nchunks; ++i) {
        slots[2 * i] = out[i].start;
        slots[2 * i + 1] = out[i].end;
    }
    DevBuf d_slots, d_vals;
    CU_TRY(ctx, d_slots.alloc(slots.size() * 8, ctx->stream));
    CU_TRY(ctx, d_vals.alloc(slots.size() * 8, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(d_slots.p, slots.data(), slots.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    CU_TRY(ctx, launch_gather_slots(idx->d_entries, idx->entry_bytes, idx->len, d_slots.as<uint64_t>(), slots.size(),
                                    d_vals.as<uint64_t>(), ctx->stream));
    ctx->launches += 1;
    CU_TRY(ctx, cudaMemcpyAsync(vals.data(), d_vals.p, slots.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < nchunks; ++i) {
        out[i].byte_start = vals[2 * i] == UINT64_MAX ? UINT64_MAX : vals[2 * i] + 1;
        out[i].byte_end = vals[2 * i + 1] == UINT64_MAX ? UINT64_MAX : vals[2 * i + 1] + 1;
    }
    return CSVB200_OK;
}

static int seek_device(csvb200_index* idx, const uint32_t* d_rec, const uint32_t* d_fld, size_t nq,
                       csvb200_range* d_out, uint32_t* d_oob)
{
    csvb200_ctx* ctx = idx->ctx;
    LookupParams p{};
    p.index = idx->d_entries;
    p.entry_bytes = idx->entry_bytes;
    p.index_len = idx->len;
    p.record_cnt = idx->record_cnt;
    p.field_cnt = idx->field_cnt;
    p.row_size = (uint32_t)idx->jump;
    p.rec = d_rec;
    p.fld = d_fld;
    p.nq = nq;
    p.ranges = reinterpret_cast<uint64_t*>(d_out);
    p.oob = d_oob;
    CU_TRY(ctx, launch_seek(p, ctx->stream));
    if (nq) ctx->launches += 1;
    return CSVB200_OK;
}

static int seek_prepare(csvb200_index* idx)
{
    if (!idx) return CSVB200_ERR_INVALID_ARG;
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    if (!idx->tape_ready)  // RecordSource::record_cnt() == None -> InvalidState (record_source.rs:77-79)
        return fail(idx->ctx, CSVB200_ERR_INVALID_STATE, "csvb200_tape_init has not been called");
    CU_TRY(idx->ctx, cudaSetDevice(idx->ctx->device));
    return CSVB200_OK;
}

// Host arrays in / out.  Queries go up and ranges come down in chunks of kSeekChunk queries on two
// streams (H2D + kernel on the context's stream, D2H on the copy stream), double buffered, so a large
// batch costs about max(up, down) of PCIe time instead of their sum plus the kernel.  Pinned caller
// arrays (csvb200_host_alloc) are DMA'd in place; pageable ones are staged through pinned buffers.
static int seek_host(csvb200_index* idx, const uint32_t* rec, const uint32_t* fld, size_t nq, csvb200_range* out)
{
    int rc = seek_prepare(idx);
    if (rc) return rc;
    if (nq == 0) return CSVB200_OK;
    if (!rec || !out) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    csvb200_ctx* ctx = idx->ctx;
    constexpr size_t kSeekChunk = 1u << 20;
    const size_t chunk = std::min(nq, kSeekChunk);
    const size_t nchunks = (nq + chunk - 1) / chunk;
    const int nslots = nchunks > 1 ? 2 : 1;
    // small batches (and the scalar seeks) skip the staging allocation: the driver stages tiny pageable copies itself
    const bool direct = nq <= 4096 || (is_pinned(rec) && is_pinned(out) && (!fld || is_pinned(fld)));
    cudaStream_t s_up = ctx->stream, s_down = nchunks > 1 ? ctx->copy_stream : ctx->stream;

    uint32_t *d_rec = nullptr, *d_fld = nullptr, *d_oob = nullptr;
    csvb200_range* d_out = nullptr;
    uint8_t* h_stage = nullptr;  // per slot: [rec chunk][fld chunk][out chunk]
    const size_t slot_bytes = chunk * (2 * sizeof(uint32_t) + sizeof(csvb200_range));
    cudaEvent_t k_done[2] = {nullptr, nullptr}, d_done[2] = {nullptr, nullptr};
    uint32_t oob = 0;
    auto cleanup = [&]() {
        cudaStreamSynchronize(s_down);
        cudaStreamSynchronize(s_up);
        if (d_rec) cudaFreeAsync(d_rec, s_up);
        if (d_fld) cudaFreeAsync(d_fld, s_up);
        if (d_out) cudaFreeAsync(d_out, s_up);
        if (d_oob) cudaFreeAsync(d_oob, s_up);
        for (int i = 0; i < 2; ++i) {
            if (k_done[i]) cudaEventDestroy(k_done[i]);
            if (d_done[i]) cudaEventDestroy(d_done[i]);
        }
        cudaGetLastError();
    };
#define SEEK_TRY(expr)                                                                                     \
    do {                                                                                                   \
        cudaError_t e_ = (expr);                                                                           \
        if (e_ != cudaSuccess) {                                                                           \
            cudaGetLastError();                                                                            \
            cleanup();                                                                                     \
            return fail(ctx, e_ == cudaErrorMemoryAllocation ? CSVB200_ERR_OOM : CSVB200_ERR_CUDA,         \
                        std::string(#expr) + ": " + cudaGetErrorString(e_));                               \
        }                                                                                                  \
    } while (0)
    SEEK_TRY(pool_malloc((void**)&d_rec, nslots * chunk * sizeof(uint32_t), s_up));
    if (fld) SEEK_TRY(pool_malloc((void**)&d_fld, nslots * chunk * sizeof(uint32_t), s_up));
    SEEK_TRY(pool_malloc((void**)&d_out, nslots * chunk * sizeof(csvb200_range), s_up));
    SEEK_TRY(pool_malloc((void**)&d_oob, sizeof(uint32_t), s_up));
    SEEK_TRY(cudaMemsetAsync(d_oob, 0, sizeof(uint32_t), s_up));
    if (!direct) {
        if (ctx->seek_stage_bytes < nslots * slot_bytes) {   // page-locking is slow: keep the buffer in the context
            if (ctx->h_seek_stage) cudaFreeHost(ctx->h_seek_stage);
            ctx->h_seek_stage = nullptr;
            ctx->seek_stage_bytes = 0;
            SEEK_TRY(cudaHostAlloc((void**)&ctx->h_seek_stage, nslots * slot_bytes, cudaHostAllocDefault));
            ctx->seek_stage_bytes = nslots * slot_bytes;
        }
        h_stage = ctx->h_seek_stage;
    }
    for (int i = 0; i < nslots; ++i) {
        SEEK_TRY(cudaEventCreateWithFlags(&k_done[i], cudaEventDisableTiming));
        SEEK_TRY(cudaEventCreateWithFlags(&d_done[i], cudaEventDisableTiming));
    }
    auto stage_rec = [&](int slot) { return reinterpret_cast<uint32_t*>(h_stage + slot * slot_bytes); };
    auto stage_fld = [&](int slot) { return stage_rec(slot) + chunk; };
    auto stage_out = [&](int slot) { return reinterpret_cast<csvb200_range*>(stage_fld(slot) + chunk); };
    // drain slot: (staged mode) wait for its D2H and hand the ranges of chunk c to the caller's array
    auto drain = [&](size_t c) -> cudaError_t {
        const int slot = (int)(c % nslots);
        cudaError_t e = cudaEventSynchronize(d_done[slot]);
        if (e == cudaSuccess && !direct) {
            const size_t off = c * chunk, len = std::min(chunk, nq - off);
            std::memcpy(out + off, stage_out(slot), len * sizeof(csvb200_range));
        }
        return e;
    };
    for (size_t c = 0; c < nchunks; ++c) {
        const int slot = (int)(c % nslots);
        const size_t off = c * chunk, len = std::min(chunk, nq - off);
        if (c >= (size_t)nslots) {
            if (!direct) SEEK_TRY(drain(c - nslots));                 // frees the slot's staging buffers
            SEEK_TRY(cudaStreamWaitEvent(s_up, d_done[slot], 0));    // and its device output buffer
        }
        const uint32_t* src_rec = rec + off;
        const uint32_t* src_fld = fld ? fld + off : nullptr;
        if (!direct) {
            std::memcpy(stage_rec(slot), src_rec, len * sizeof(uint32_t));
            src_rec = stage_rec(slot);
            if (fld) {
                std::memcpy(stage_fld(slot), src_fld, len * sizeof(uint32_t));
                src_fld = stage_fld(slot);
            }
        }
        uint32_t* dr = d_rec + slot * chunk;
        uint32_t* df = fld ? d_fld + slot * chunk : nullptr;
        csvb200_range* dout = d_out + slot * chunk;
        SEEK_TRY(cudaMemcpyAsync(dr, src_rec, len * sizeof(uint32_t), cudaMemcpyHostToDevice, s_up));
        if (fld) SEEK_TRY(cudaMemcpyAsync(df, src_fld, len * sizeof(uint32_t), cudaMemcpyHostToDevice, s_up));
        rc = seek_device(idx, dr, df, len, dout, d_oob);
        if (rc) {
            cleanup();
            return rc;
        }
        SEEK_TRY(cudaEventRecord(k_done[slot], s_up));
        if (s_down != s_up) SEEK_TRY(cudaStreamWaitEvent(s_down, k_done[slot], 0));
        SEEK_TRY(cudaMemcpyAsync(direct ? out + off : stage_out(slot), dout, len * sizeof(csvb200_range),
                                 cudaMemcpyDeviceToHost, s_down));
        SEEK_TRY(cudaEventRecord(d_done[slot], s_down));
    }
    for (size_t c = nchunks > (size_t)nslots ? nchunks - nslots : 0; c < nchunks; ++c) SEEK_TRY(drain(c));
    SEEK_TRY(cudaStreamSynchronize(s_down));
    SEEK_TRY(cudaMemcpyAsync(&oob, d_oob, sizeof(uint32_t), cudaMemcpyDeviceToHost, s_up));
    SEEK_TRY(cudaStreamSynchronize(s_up));
#undef SEEK_TRY
    cleanup();
    if (oob) return fail(ctx, CSVB200_ERR_OUT_OF_BOUNDS, "lookup slot past the end of the index");
    return CSVB200_OK;
}

int csvb200_seek_records(csvb200_index* idx, const uint32_t* rec, size_t nq, csvb200_range* out)
{
    return seek_host(idx, rec, nullptr, nq, out);
}

int csvb200_seek_fields(csvb200_index* idx, const uint32_t* rec, const uint32_t* fld, size_t nq, csvb200_range* out)
{
    if (idx && nq && !fld) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    return seek_host(idx, rec, fld, nq, out);
}

int csvb200_seek_record(csvb200_index* idx, uint32_t record_idx, csvb200_range* out, int* found)
{
    if (!out || !found) return CSVB200_ERR_INVALID_ARG;
    int rc = seek_host(idx, &record_idx, nullptr, 1, out);
    if (!rc) *found = out->start != UINT64_MAX;
    return rc;
}

int csvb200_seek_field(csvb200_index* idx, uint32_t record_idx, uint32_t field_idx, csvb200_range* out, int* found)
{
    if (!out || !found) return CSVB200_ERR_INVALID_ARG;
    int rc = seek_host(idx, &record_idx, &field_idx, 1, out);
    if (!rc) *found = out->start != UINT64_MAX;
    return rc;
}

int csvb200_seek_fields_device(csvb200_index* idx, const uint32_t* d_rec, const uint32_t* d_fld, size_t nq,
                               csvb200_range* d_out)
{
    int rc = seek_prepare(idx);
    if (rc) return rc;
    if (nq && (!d_rec || !d_fld || !d_out)) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    // out-of-bounds slots are reported as None on this asynchronous path
    return seek_device(idx, d_rec, d_fld, nq, d_out, reinterpret_cast<uint32_t*>(idx->ctx->d_cells + (kCells - 1) * kCellWords));
}

int csvb200_seek_records_device(csvb200_index* idx, const uint32_t* d_rec, size_t nq, csvb200_range* d_out)
{
    int rc = seek_prepare(idx);
    if (rc) return rc;
    if (nq && (!d_rec || !d_out)) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    return seek_device(idx, d_rec, nullptr, nq, d_out, reinterpret_cast<uint32_t*>(idx->ctx->d_cells + (kCells - 1) * kCellWords));
}

static int values_prepare(csvb200_index* idx)
{
    int rc = seek_prepare(idx);
    if (rc) return rc;
    if (!idx->d_bytes_owned && !idx->src)
        return fail(idx->ctx, CSVB200_ERR_INVALID_STATE, "index was built without CSVB200_BUILD_KEEP_BYTES");
    return CSVB200_OK;
}

static int values_args(csvb200_index* idx, const void* rec, const void* fld, size_t nq, uint32_t flags, const void* offsets)
{
    if (!offsets || (nq && !rec)) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    if (flags & ~(CSVB200_FIELD_UNQUOTE | CSVB200_FIELD_TRIM)) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "unknown field flags");
    if (flags && !fld) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "flags apply to fields only (fld == NULL: records)");
    return CSVB200_OK;
}

static ValuesParams values_params(const csvb200_index* idx, const uint32_t* rec, const uint32_t* fld, size_t nq, uint32_t flags)
{
    ValuesParams p{};
    p.index_len = idx->len;
    p.record_cnt = idx->record_cnt;
    p.field_cnt = idx->field_cnt;
    p.row_size = (uint32_t)idx->jump;
    p.flags = flags;
    p.rec = rec;
    p.fld = fld;
    p.nq = nq;
    return p;
}

static ValuesLocal values_source(const csvb200_index* idx)
{
    return ValuesLocal{idx->d_entries, idx->entry_bytes, idx->d_bytes_owned ? idx->d_bytes_owned : idx->src, idx->n, idx->pos_bias};
}

}  // extern "C"

namespace csvb200 {

int values_enqueue(csvb200_ctx* ctx, ValuesParams p, const ValuesLocal* local, const SegmentTable* seg, const ShardBytes* sb,
                   bool write_pass)
{
    const size_t sbytes = values_scratch_bytes(p.nq);
    int rc = ensure_scratch(ctx, sbytes);
    if (rc) return rc;
    CU_TRY(ctx, cudaMemsetAsync(ctx->d_scratch, 0, sbytes, ctx->stream));
    p.ticket = reinterpret_cast<uint32_t*>(ctx->d_scratch);
    p.tile_desc = reinterpret_cast<uint64_t*>(ctx->d_scratch + 128);
    if (p.nq == 0) {   // every caller of an empty batch asks for offsets that start at 0
        CU_TRY(ctx, cudaMemsetAsync(p.offsets, 0, sizeof(uint64_t), ctx->stream));
        return CSVB200_OK;
    }
    CU_TRY(ctx, local ? launch_values_offsets(p, *local, ctx->stream) : launch_values_offsets_sharded(p, *seg, *sb, ctx->stream));
    ctx->launches += 1;
    if (write_pass && p.out) {
        CU_TRY(ctx, local ? launch_values_write(p, *local, ctx->stream) : launch_values_write_sharded(p, *seg, *sb, ctx->stream));
        ctx->launches += 1;
    }
    return CSVB200_OK;
}

}  // namespace csvb200

extern "C" {

// Host arrays in / out, in chunks of kValuesChunk queries.  Sweep 1: per chunk, the queries go up, the offsets pass
// runs with the running total as its base, and the offsets and found bits come down in place; the counters decide
// OUT_OF_BOUNDS and the total decides CAPACITY before anything is written.  Sweep 2: per chunk, the values are written
// into one device buffer sized by the largest chunk's values and go down to their place in `out`.
int csvb200_seek_values(csvb200_index* idx, const uint32_t* rec, const uint32_t* fld, size_t nq, uint32_t flags,
                        uint64_t* out_offsets, uint8_t* out, size_t out_cap, size_t* out_len, uint64_t* found_bits)
{
    int rc = values_prepare(idx);
    if (rc) return rc;
    csvb200_ctx* ctx = idx->ctx;
    if (!out_len) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    rc = values_args(idx, rec, fld, nq, flags, out_offsets);
    if (rc) return rc;
    *out_len = 0;
    out_offsets[0] = 0;
    if (nq == 0) return CSVB200_OK;
    constexpr size_t kValuesChunk = 1u << 20;   // a multiple of 64: every chunk writes whole found-bit words
    const size_t chunk = std::min(nq, kValuesChunk);
    const size_t nchunks = (nq + chunk - 1) / chunk;
    DevBuf d_rec, d_fld, d_off, d_found, d_cnt, d_out;
    CU_TRY(ctx, d_rec.alloc(chunk * sizeof(uint32_t), ctx->stream));
    if (fld) CU_TRY(ctx, d_fld.alloc(chunk * sizeof(uint32_t), ctx->stream));
    CU_TRY(ctx, d_off.alloc((chunk + 1) * sizeof(uint64_t), ctx->stream));
    if (found_bits) CU_TRY(ctx, d_found.alloc((chunk + 63) / 64 * sizeof(uint64_t), ctx->stream));
    CU_TRY(ctx, d_cnt.alloc(2 * sizeof(uint32_t), ctx->stream));
    CU_TRY(ctx, cudaMemsetAsync(d_cnt.p, 0, 2 * sizeof(uint32_t), ctx->stream));
    const ValuesLocal src = values_source(idx);
    auto upload_queries = [&](size_t off, size_t len) -> int {
        CU_TRY(ctx, cudaMemcpyAsync(d_rec.p, rec + off, len * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        if (fld) CU_TRY(ctx, cudaMemcpyAsync(d_fld.p, fld + off, len * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
        return CSVB200_OK;
    };
    uint64_t total = 0, largest = 0;
    for (size_t c = 0; c < nchunks; ++c) {
        const size_t off = c * chunk, len = std::min(chunk, nq - off);
        rc = upload_queries(off, len);
        if (rc) return rc;
        ValuesParams p = values_params(idx, d_rec.as<uint32_t>(), fld ? d_fld.as<uint32_t>() : nullptr, len, flags);
        p.offsets = d_off.as<uint64_t>();
        p.offset_base = total;
        p.found = found_bits ? d_found.as<uint32_t>() : nullptr;
        p.counts = d_cnt.as<uint32_t>();
        rc = values_enqueue(ctx, p, &src, nullptr, nullptr, false);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemcpyAsync(out_offsets + off, d_off.p, (len + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (found_bits)
            CU_TRY(ctx, cudaMemcpyAsync(found_bits + off / 64, d_found.p, (len + 63) / 64 * sizeof(uint64_t), cudaMemcpyDeviceToHost,
                                        ctx->stream));
        CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        largest = std::max<uint64_t>(largest, out_offsets[off + len] - total);
        total = out_offsets[off + len];
    }
    uint32_t counts[2] = {0, 0};
    CU_TRY(ctx, cudaMemcpyAsync(counts, d_cnt.p, sizeof(counts), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (counts[0]) return fail(ctx, CSVB200_ERR_OUT_OF_BOUNDS, "lookup slot past the end of the index");
    // positions are global; the bytes this index object holds are [pos_bias, pos_bias + n) (a shard of a sharded build)
    if (counts[1]) return fail(ctx, CSVB200_ERR_OUT_OF_BOUNDS, "value lies outside the bytes this index object holds (another shard)");
    *out_len = (size_t)total;
    if (total > out_cap) return fail(ctx, CSVB200_ERR_CAPACITY, "values destination too small");
    if (total == 0) return CSVB200_OK;
    if (!out) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    CU_TRY(ctx, d_out.alloc(largest, ctx->stream));
    for (size_t c = 0; c < nchunks; ++c) {
        const size_t off = c * chunk, len = std::min(chunk, nq - off);
        const uint64_t base = out_offsets[off], bytes = out_offsets[off + len] - base;
        if (bytes == 0) continue;
        if (nchunks > 1) {   // one chunk: its queries and offsets are still on the device
            rc = upload_queries(off, len);
            if (rc) return rc;
            CU_TRY(ctx, cudaMemcpyAsync(d_off.p, out_offsets + off, (len + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
        }
        ValuesParams p = values_params(idx, d_rec.as<uint32_t>(), fld ? d_fld.as<uint32_t>() : nullptr, len, flags);
        p.offsets = d_off.as<uint64_t>();
        p.offset_base = base;
        p.out = d_out.as<uint8_t>();
        p.out_cap = bytes;
        CU_TRY(ctx, launch_values_write(p, src, ctx->stream));
        ctx->launches += 1;
        CU_TRY(ctx, cudaMemcpyAsync(out + base, d_out.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return CSVB200_OK;
}

int csvb200_seek_values_device(csvb200_index* idx, const uint32_t* d_rec, const uint32_t* d_fld, size_t nq, uint32_t flags,
                               uint64_t* d_offsets, uint8_t* d_out, size_t out_cap, uint64_t* d_found_bits)
{
    int rc = values_prepare(idx);
    if (rc) return rc;
    rc = values_args(idx, d_rec, d_fld, nq, flags, d_offsets);
    if (rc) return rc;
    ValuesParams p = values_params(idx, d_rec, d_fld, nq, flags);
    p.offsets = d_offsets;
    p.out = d_out;
    p.out_cap = out_cap;
    p.found = reinterpret_cast<uint32_t*>(d_found_bits);
    // out-of-bounds slots are reported as None on this asynchronous path
    p.counts = reinterpret_cast<uint32_t*>(idx->ctx->d_cells + (kCells - 1) * kCellWords);
    const ValuesLocal src = values_source(idx);
    return values_enqueue(idx->ctx, p, &src, nullptr, nullptr, true);
}

// the values of flags == 0: the old two-kernel gather (ranges to the host, a serial prefix sum there, ranges and
// offsets back up) is the same computation as the raw form of csvb200_seek_values
int csvb200_gather_fields(csvb200_index* idx, const uint32_t* rec, const uint32_t* fld, size_t nq,
                          uint64_t* out_offsets, uint8_t* out, size_t out_cap)
{
    int rc = values_prepare(idx);
    if (rc) return rc;
    if (!out_offsets || (nq && (!rec || !fld))) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    out_offsets[0] = 0;
    if (nq == 0) return CSVB200_OK;
    size_t len = 0;
    return csvb200_seek_values(idx, rec, fld, nq, CSVB200_FIELD_RAW, out_offsets, out, out_cap, &len, nullptr);
}

// enqueue lengths + scan (+ write when d_out != nullptr) of one column on the context's stream
static int materialize_enqueue(csvb200_ctx* ctx, const MatSource& src, uint32_t field_idx, uint32_t first_record, uint32_t nrec,
                               uint32_t flags, uint64_t* d_offsets, uint8_t* d_out, size_t out_cap, uint64_t offset_base,
                               bool offsets_pass, bool write_pass)
{
    MaterializeParams p{};
    p.index = src.index;
    p.entry_bytes = src.entry_bytes;
    p.index_len = src.index_len;
    p.bytes = src.bytes;
    p.n = src.n;
    p.pos_bias = src.pos_bias;
    p.record_cnt = src.record_cnt;
    p.field_cnt = src.field_cnt;
    p.row_size = src.row_size;
    p.field_idx = field_idx;
    p.first_record = first_record;
    p.nrec = nrec;
    p.flags = flags;
    p.offsets = d_offsets;
    p.out = d_out;
    p.out_cap = out_cap;
    p.offset_base = offset_base;
    if (offsets_pass) {
        const size_t sbytes = materialize_scratch_bytes(nrec);
        int rc = ensure_scratch(ctx, sbytes);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemsetAsync(ctx->d_scratch, 0, sbytes, ctx->stream));
        p.ticket = reinterpret_cast<uint32_t*>(ctx->d_scratch);
        p.tile_desc = reinterpret_cast<uint64_t*>(ctx->d_scratch + 128);
        if (nrec == 0) CU_TRY(ctx, cudaMemsetAsync(d_offsets, 0, sizeof(uint64_t), ctx->stream));
        CU_TRY(ctx, launch_materialize_offsets(p, ctx->stream));
        if (nrec) ctx->launches += 1;
    }
    if (write_pass && nrec) {
        CU_TRY(ctx, launch_materialize_write(p, ctx->stream));
        ctx->launches += 1;
    }
    return CSVB200_OK;
}

static int materialize_prepare(csvb200_index* idx, uint32_t flags)
{
    int rc = seek_prepare(idx);
    if (rc) return rc;
    if (flags & ~(CSVB200_FIELD_UNQUOTE | CSVB200_FIELD_TRIM)) return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "unknown field flags");
    if (!idx->d_bytes_owned && !idx->src && idx->n)
        return fail(idx->ctx, CSVB200_ERR_INVALID_STATE, "index was built without CSVB200_BUILD_KEEP_BYTES");
    return CSVB200_OK;
}

static MatSource source_of(const csvb200_index* idx)
{
    return MatSource{idx->d_entries, idx->len, idx->d_bytes_owned ? idx->d_bytes_owned : idx->src, idx->n, idx->pos_bias,
                     idx->record_cnt, idx->field_cnt, (uint32_t)idx->jump, idx->entry_bytes};
}

}  // extern "C"

namespace csvb200 {

// several columns, one sweep per pass (materialize.cu: a thread owns a row and walks its requested fields)
int materialize_multi_enqueue(csvb200_ctx* ctx, const MatSource& src, const uint32_t* fields, uint32_t ncols,
                              uint32_t first_record, uint32_t nrec, uint32_t flags, uint64_t* const* d_offsets,
                              uint8_t* const* d_outs, const size_t* out_caps, const uint64_t* offset_base, bool offsets_pass,
                              bool write_pass)
{
    if (ncols == 1)   // one column: the single-column kernels (1024-record tiles) are the faster form
        return materialize_enqueue(ctx, src, fields[0], first_record, nrec, flags, d_offsets[0], d_outs ? d_outs[0] : nullptr,
                                   out_caps ? out_caps[0] : 0, offset_base ? offset_base[0] : 0, offsets_pass, write_pass);
    // The multi-column kernels keep lengths and tile totals in u32.  Up to 4 GiB that is exact: one column's values over
    // distinct records are disjoint slices of the input without their line ends, so a tile's total stays below 2^32.
    // Past 4 GiB a value or a tile can reach 2^32: the columns go one after the other through the u64 kernels.
    if (src.n > UINT32_MAX) {
        for (uint32_t c = 0; c < ncols; ++c) {
            int rc = materialize_enqueue(ctx, src, fields[c], first_record, nrec, flags, d_offsets[c],
                                         d_outs ? d_outs[c] : nullptr, out_caps ? out_caps[c] : 0,
                                         offset_base ? offset_base[c] : 0, offsets_pass, write_pass);
            if (rc) return rc;
        }
        return CSVB200_OK;
    }
    MaterializeMultiParams p{};
    p.index = src.index;
    p.entry_bytes = src.entry_bytes;
    p.index_len = src.index_len;
    p.bytes = src.bytes;
    p.n = src.n;
    p.pos_bias = src.pos_bias;
    p.record_cnt = src.record_cnt;
    p.field_cnt = src.field_cnt;
    p.row_size = src.row_size;
    p.first_record = first_record;
    p.nrec = nrec;
    p.flags = flags;
    p.ncols = ncols;
    p.tiles = (nrec + kMultiThreads - 1) / kMultiThreads;
    for (uint32_t c = 0; c < ncols; ++c) {
        p.field_idx[c] = fields[c];
        p.offsets[c] = d_offsets[c];
        p.out[c] = d_outs ? d_outs[c] : nullptr;
        p.out_cap[c] = out_caps ? out_caps[c] : 0;
        p.offset_base[c] = offset_base ? offset_base[c] : 0;
    }
    if (offsets_pass) {
        const size_t sbytes = materialize_multi_scratch_bytes(nrec, ncols);
        int rc = ensure_scratch(ctx, sbytes);
        if (rc) return rc;
        CU_TRY(ctx, cudaMemsetAsync(ctx->d_scratch, 0, sbytes, ctx->stream));
        p.ticket = reinterpret_cast<uint32_t*>(ctx->d_scratch);
        p.tile_desc = reinterpret_cast<uint64_t*>(ctx->d_scratch + 128);
        if (nrec == 0)
            for (uint32_t c = 0; c < ncols; ++c) CU_TRY(ctx, cudaMemsetAsync(d_offsets[c], 0, sizeof(uint64_t), ctx->stream));
        CU_TRY(ctx, launch_materialize_multi_offsets(p, ctx->stream));
        if (nrec) ctx->launches += 1;
    }
    if (write_pass && nrec) {
        CU_TRY(ctx, launch_materialize_multi_write(p, ctx->stream));
        ctx->launches += 1;
    }
    return CSVB200_OK;
}

}  // namespace csvb200

extern "C" {

int csvb200_materialize_columns_device(csvb200_index* idx, const uint32_t* fields, uint32_t ncols, uint32_t first_record,
                                       uint32_t nrec, uint32_t flags, uint64_t* const* d_offsets, uint8_t* const* d_outs,
                                       const size_t* out_caps)
{
    int rc = materialize_prepare(idx, flags);
    if (rc) return rc;
    if (!fields || !d_offsets || ncols == 0 || ncols > kMatMaxCols)
        return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "1 <= ncols <= 32 and non-null arrays");
    for (uint32_t c = 0; c < ncols; ++c)
        if (!d_offsets[c] || (out_caps && out_caps[c] && (!d_outs || !d_outs[c])))
            return fail(idx->ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    return materialize_multi_enqueue(idx->ctx, source_of(idx), fields, ncols, first_record, nrec, flags, d_offsets, d_outs,
                                     out_caps, nullptr, true, d_outs != nullptr);
}

int csvb200_materialize_columns(csvb200_index* idx, const uint32_t* fields, uint32_t ncols, uint32_t first_record,
                                uint32_t nrec, uint32_t flags, uint64_t* const* out_offsets, uint8_t* const* outs,
                                const size_t* out_caps, size_t* out_lens)
{
    int rc = materialize_prepare(idx, flags);
    if (rc) return rc;
    csvb200_ctx* ctx = idx->ctx;
    if (!fields || !out_offsets || !out_lens || ncols == 0 || ncols > kMatMaxCols)
        return fail(ctx, CSVB200_ERR_INVALID_ARG, "1 <= ncols <= 32 and non-null arrays");
    std::vector<DevBuf> d_off(ncols), d_out(ncols);
    std::vector<uint64_t*> p_off(ncols);
    std::vector<uint8_t*> p_out(ncols, nullptr);
    std::vector<size_t> caps(ncols, 0);
    for (uint32_t c = 0; c < ncols; ++c) {
        if (!out_offsets[c]) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
        CU_TRY(ctx, d_off[c].alloc(((size_t)nrec + 1) * sizeof(uint64_t), ctx->stream));
        p_off[c] = d_off[c].as<uint64_t>();
    }
    rc = materialize_multi_enqueue(ctx, source_of(idx), fields, ncols, first_record, nrec, flags, p_off.data(), nullptr, nullptr,
                                   nullptr, true, false);
    if (rc) return rc;
    for (uint32_t c = 0; c < ncols; ++c)
        CU_TRY(ctx, cudaMemcpyAsync(out_offsets[c], p_off[c], ((size_t)nrec + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    bool small = false, any = false;
    for (uint32_t c = 0; c < ncols; ++c) {
        const uint64_t total = out_offsets[c][nrec];
        out_lens[c] = (size_t)total;
        if (total > (out_caps ? out_caps[c] : 0)) small = true;
        if (total) any = true;
    }
    if (small) return fail(ctx, CSVB200_ERR_CAPACITY, "materialize destination too small");
    if (!any) return CSVB200_OK;
    if (!outs) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    for (uint32_t c = 0; c < ncols; ++c) {
        if (out_lens[c] && !outs[c]) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
        CU_TRY(ctx, d_out[c].alloc(out_lens[c], ctx->stream));
        p_out[c] = d_out[c].as<uint8_t>();
        caps[c] = out_lens[c];
    }
    rc = materialize_multi_enqueue(ctx, source_of(idx), fields, ncols, first_record, nrec, flags, p_off.data(), p_out.data(),
                                   caps.data(), nullptr, false, true);
    if (rc) return rc;
    for (uint32_t c = 0; c < ncols; ++c)
        if (out_lens[c]) CU_TRY(ctx, cudaMemcpyAsync(outs[c], p_out[c], out_lens[c], cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return CSVB200_OK;
}

int csvb200_materialize_column_device(csvb200_index* idx, uint32_t field_idx, uint32_t first_record, uint32_t nrec,
                                      uint32_t flags, uint64_t* d_offsets, uint8_t* d_out, size_t out_cap)
{
    return csvb200_materialize_columns_device(idx, &field_idx, 1, first_record, nrec, flags, &d_offsets, d_out ? &d_out : nullptr,
                                              &out_cap);
}

int csvb200_materialize_column(csvb200_index* idx, uint32_t field_idx, uint32_t first_record, uint32_t nrec,
                               uint32_t flags, uint64_t* out_offsets, uint8_t* out, size_t out_cap, size_t* out_len)
{
    return csvb200_materialize_columns(idx, &field_idx, 1, first_record, nrec, flags, &out_offsets, &out, &out_cap, out_len);
}

int csvb200_validate_utf8_device(csvb200_ctx* ctx, const void* dev_bytes, size_t n, uint64_t* d_result)
{
    if (!ctx || !d_result || (n && !dev_bytes)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaMemsetAsync(d_result, 0xff, sizeof(uint64_t), ctx->stream));
    CU_TRY(ctx, cudaMemsetAsync(d_result + 1, 0, sizeof(uint64_t), ctx->stream));
    CU_TRY(ctx, launch_utf8_validate(static_cast<const uint8_t*>(dev_bytes), n, d_result, ctx->stream));
    if (n) ctx->launches += 1;
    return CSVB200_OK;
}

int csvb200_validate_utf8(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* valid_up_to, int* is_ascii)
{
    if (!ctx || (n && !host_bytes)) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    DevBuf d_buf;
    CU_TRY(ctx, d_buf.alloc(n + 16, ctx->stream));
    uint8_t* d_in = d_buf.as<uint8_t>();
    int rc = upload(ctx, d_in, host_bytes, n);
    CellLease lease(ctx, 1);
    if (!lease.ok()) return fail(ctx, CSVB200_ERR_OOM, "no free result cell (4095 live index objects)");
    const size_t cell = lease.first;
    uint64_t* d_cell = ctx->d_cells + cell * kCellWords;
    uint64_t* h_cell = ctx->h_cells + cell * kCellWords;
    if (!rc) rc = csvb200_validate_utf8_device(ctx, d_in, n, d_cell);
    if (!rc) {
        CU_TRY(ctx, cudaMemcpyAsync(h_cell, d_cell, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        if (valid_up_to) *valid_up_to = h_cell[0];
        if (is_ascii) *is_ascii = h_cell[1] ? 0 : 1;
    }
    return rc;
}

// ---- on-disk index (SURVEY 8f rank 4): 64-byte little-endian header + the u64 entries ----------------
namespace {
struct IndexFileHeader {
    char magic[8];          // "CSVB2IDX"
    uint32_t version;       // 1
    uint32_t flags;         // bit 0: Tape metadata present, bit 1: CRLF
    uint64_t input_bytes;
    uint64_t entries;
    uint32_t field_cnt;
    uint32_t record_cnt;
    uint64_t jump;
    uint64_t end_parity;
    uint64_t checksum;      // wrapping sum of the entries
};
static_assert(sizeof(IndexFileHeader) == 64, "on-disk header is 64 bytes");
const char kIndexMagic[8] = {'C', 'S', 'V', 'B', '2', 'I', 'D', 'X'};
}  // namespace

int csvb200_index_save(csvb200_index* idx, const char* path)
{
    if (!idx || !path) return CSVB200_ERR_INVALID_ARG;
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    csvb200_ctx* ctx = idx->ctx;
    std::vector<uint64_t> host;
    try {
        host.resize(idx->len);
    } catch (const std::exception&) {
        return fail(ctx, CSVB200_ERR_OOM, "index does not fit in host memory");
    }
    rc = csvb200_index_copy_out(idx, host.data(), host.size());
    if (rc) return rc;
    IndexFileHeader h{};
    std::memcpy(h.magic, kIndexMagic, 8);
    h.version = 1;
    h.flags = (idx->tape_ready ? 1u : 0u) | (idx->crlf ? 2u : 0u);
    h.input_bytes = idx->n;
    h.entries = idx->len;
    h.field_cnt = idx->field_cnt;
    h.record_cnt = idx->record_cnt;
    h.jump = idx->jump;
    h.end_parity = (uint64_t)idx->end_parity;
    for (uint64_t v : host) h.checksum += v;
    FILE* f = std::fopen(path, "wb");
    if (!f) return fail(ctx, CSVB200_ERR_IO, std::string("open ") + path + ": " + std::strerror(errno));
    const bool ok = std::fwrite(&h, sizeof(h), 1, f) == 1 &&
                    (host.empty() || std::fwrite(host.data(), sizeof(uint64_t), host.size(), f) == host.size());
    const bool closed = std::fclose(f) == 0;
    if (!ok || !closed) return fail(ctx, CSVB200_ERR_IO, std::string("write ") + path + " failed");
    return CSVB200_OK;
}

int csvb200_index_load(csvb200_ctx* ctx, const char* path, csvb200_index** out)
{
    if (!ctx || !path || !out) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    FILE* f = std::fopen(path, "rb");
    if (!f) return fail(ctx, CSVB200_ERR_IO, std::string("open ") + path + ": " + std::strerror(errno));
    IndexFileHeader h{};
    std::vector<uint64_t> host;
    bool ok = std::fread(&h, sizeof(h), 1, f) == 1 && std::memcmp(h.magic, kIndexMagic, 8) == 0 && h.version == 1;
    if (ok) {
        std::fseek(f, 0, SEEK_END);
        const long long size = std::ftell(f);
        // entries is bounded by the file size BEFORE it is multiplied (a huge value must not wrap)
        ok = size >= (long long)sizeof(h) && h.entries >= 1 &&
             h.entries <= ((unsigned long long)size - sizeof(h)) / sizeof(uint64_t) &&
             (unsigned long long)size == sizeof(h) + h.entries * sizeof(uint64_t);
        std::fseek(f, (long)sizeof(h), SEEK_SET);
    }
    if (ok) {
        try {
            host.resize(h.entries);
        } catch (const std::exception&) {   // nothing may unwind across the C ABI
            std::fclose(f);
            return fail(ctx, CSVB200_ERR_OOM, std::string(path) + ": index does not fit in host memory");
        }
        ok = std::fread(host.data(), sizeof(uint64_t), host.size(), f) == host.size();
    }
    std::fclose(f);
    uint64_t sum = 0;
    for (uint64_t v : host) sum += v;
    if (!ok || host.empty() || sum != h.checksum || host[0] != 0)
        return fail(ctx, CSVB200_ERR_INVALID_CSV_FORMAT, std::string(path) + ": not a csvb200 index file (bad magic, size or checksum)");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    csvb200_index* idx = nullptr;
    int rc = new_index(ctx, &idx);
    if (rc) return rc;
    idx->cap = host.size();
    cudaError_t e = pool_malloc(&idx->d_entries, idx->cap * sizeof(uint64_t), ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(idx->d_entries, host.data(), host.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        csvb200_index_free(idx);
        return fail(ctx, e == cudaErrorMemoryAllocation ? CSVB200_ERR_OOM : CSVB200_ERR_CUDA, std::string("index load: ") + cudaGetErrorString(e));
    }
    idx->len = host.size();
    idx->n = h.input_bytes;
    idx->end_parity = (int)(h.end_parity & 1u);
    idx->synced = true;
    if (h.flags & 1u) {
        idx->tape_ready = true;
        idx->crlf = (h.flags & 2u) ? 1 : 0;
        idx->field_cnt = h.field_cnt;
        idx->record_cnt = h.record_cnt;
        idx->jump = h.jump;
    }
    *out = idx;
    return CSVB200_OK;
}

int csvb200_block_masks(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint64_t* quote_words,
                        uint64_t* sep_words)
{
    if (!ctx || (n && (!host_bytes || !quote_words || !sep_words))) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    if (n == 0) return CSVB200_OK;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const size_t nb = (n + 63) / 64;
    DevBuf d_in, d_q, d_s;
    CU_TRY(ctx, d_in.alloc(n, ctx->stream));
    CU_TRY(ctx, d_q.alloc(nb * 8, ctx->stream));
    CU_TRY(ctx, d_s.alloc(nb * 8, ctx->stream));
    int rc = upload(ctx, d_in.as<uint8_t>(), host_bytes, n);
    if (rc) return rc;
    CU_TRY(ctx, launch_block_masks(d_in.as<uint8_t>(), n, d_q.as<uint64_t>(), d_s.as<uint64_t>(), ctx->stream));
    ctx->launches += 1;
    CU_TRY(ctx, cudaMemcpyAsync(quote_words, d_q.p, nb * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(sep_words, d_s.p, nb * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return CSVB200_OK;
}

int csvb200_class_bytes(csvb200_ctx* ctx, const uint8_t* host_bytes, size_t n, uint8_t* out)
{
    if (!ctx || (n && (!host_bytes || !out))) return fail(ctx, CSVB200_ERR_INVALID_ARG, "null argument");
    if (n == 0) return CSVB200_OK;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    DevBuf d_in, d_out;
    CU_TRY(ctx, d_in.alloc(n, ctx->stream));
    CU_TRY(ctx, d_out.alloc(n, ctx->stream));
    int rc = upload(ctx, d_in.as<uint8_t>(), host_bytes, n);
    if (rc) return rc;
    CU_TRY(ctx, launch_class_bytes(d_in.as<uint8_t>(), n, d_out.as<uint8_t>(), ctx->stream));
    ctx->launches += 1;
    CU_TRY(ctx, cudaMemcpyAsync(out, d_out.p, n, cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return CSVB200_OK;
}

}  // extern "C"
