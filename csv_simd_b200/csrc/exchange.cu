// exchange.cu -- host side of the cross-GPU exchange (peer-mapped mailboxes, protocol in internal.h ExchangeArgs /
// index_common.cuh exchange_post_and_resolve) and the all-GPUs-of-one-process front end (csvb200_multi_*).
//
// Replaces the NCCL all-gather + verify launch of round 1 for the one thing that has to cross GPUs when a file is
// split "without first knowing record breaks" (reference README.md:24): 32 bytes per shard.  The rows travel as plain
// NVLink P2P stores issued from inside the index-build launch; this file only allocates the mailboxes, maps the
// peers' ones (CUDA IPC between processes, peer access inside one process) and offers the host-side views.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "ctx.h"
#include "record_split.h"
#include "slice_pool.h"
#include "utf8_halo.h"

using namespace csvb200;

static_assert(CSVB200_EXCHANGE_HANDLE_BYTES >= sizeof(cudaIpcMemHandle_t), "handle blob too small");
static_assert(CSVB200_EXCHANGE_MAX_WORLD == kExMaxWorld, "header / internal world limit differ");

namespace {

int upload_peer_table(csvb200_exchange* ex)
{
    csvb200_ctx* ctx = ex->ctx;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaMemcpy(ex->d_peers, ex->peer, sizeof(ex->peer), cudaMemcpyHostToDevice));
    ex->connected = true;
    return CSVB200_OK;
}

}  // namespace

extern "C" {

int csvb200_exchange_create(csvb200_ctx* ctx, uint32_t rank, uint32_t world, csvb200_exchange** out)
{
    if (!ctx || !out) return CSVB200_ERR_INVALID_ARG;
    *out = nullptr;
    if (world == 0 || world > kExMaxWorld || rank >= world)
        return fail(ctx, CSVB200_ERR_INVALID_ARG, "exchange: 1 <= world <= 16 and rank < world");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    csvb200_exchange* ex = new (std::nothrow) csvb200_exchange();
    if (!ex) return fail(ctx, CSVB200_ERR_OOM, "host allocation failed");
    ex->ctx = ctx;
    ex->rank = rank;
    ex->world = world;
    if (const char* t = std::getenv("CSVB200_EXCHANGE_TIMEOUT_MS")) {
        const long ms = std::atol(t);
        if (ms >= 1 && ms <= 600000) ex->timeout_ns = (uint64_t)ms * 1000000ull;
    }
    cudaError_t e = cudaMalloc((void**)&ex->d_mbox, kExMailboxBytes);   // cudaMalloc, not the async pool: IPC-exportable
    if (e == cudaSuccess) e = cudaMemset(ex->d_mbox, 0, kExMailboxBytes);   // epoch 0 never matches a build (epochs start at 1)
    if (e == cudaSuccess) e = cudaMalloc((void**)&ex->d_peers, sizeof(ex->peer));
    if (e == cudaSuccess) e = cudaMalloc((void**)&ex->d_row4, 4 * sizeof(uint64_t));
    if (e == cudaSuccess) e = cudaHostAlloc((void**)&ex->h_rows, kExMaxWorld * kExRowWords * sizeof(uint64_t), cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        csvb200_exchange_destroy(ex);
        return fail(ctx, e == cudaErrorMemoryAllocation ? CSVB200_ERR_OOM : CSVB200_ERR_CUDA,
                    std::string("exchange: ") + cudaGetErrorString(e));
    }
    ex->peer[rank] = ex->d_mbox;
    if (world == 1) {
        int rc = upload_peer_table(ex);
        if (rc) {
            csvb200_exchange_destroy(ex);
            return rc;
        }
    }
    *out = ex;
    return CSVB200_OK;
}

int csvb200_exchange_handle(csvb200_exchange* ex, uint8_t* out)
{
    if (!ex || !out) return CSVB200_ERR_INVALID_ARG;
    csvb200_ctx* ctx = ex->ctx;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    CU_TRY(ctx, cudaIpcGetMemHandle(&h, ex->d_mbox));
    std::memset(out, 0, CSVB200_EXCHANGE_HANDLE_BYTES);
    std::memcpy(out, &h, sizeof(h));
    return CSVB200_OK;
}

int csvb200_exchange_connect(csvb200_exchange* ex, const uint8_t* handles)
{
    if (!ex || !handles) return CSVB200_ERR_INVALID_ARG;
    csvb200_ctx* ctx = ex->ctx;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    for (uint32_t r = 0; r < ex->world; ++r) {
        if (r == ex->rank || ex->peer[r]) continue;
        cudaIpcMemHandle_t h;
        std::memcpy(&h, handles + (size_t)r * CSVB200_EXCHANGE_HANDLE_BYTES, sizeof(h));
        void* p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(ctx, CSVB200_ERR_EXCHANGE,
                        "exchange: cannot map the mailbox of rank " + std::to_string(r) + " (cudaIpcOpenMemHandle: " +
                            cudaGetErrorString(e) + "); ranks must be processes on one node with peer access");
        }
        ex->peer[r] = static_cast<uint64_t*>(p);
        ex->ipc_opened[r] = true;
    }
    return upload_peer_table(ex);
}

int csvb200_exchange_connect_local(csvb200_exchange* const* all, uint32_t world)
{
    if (!all || world == 0 || world > kExMaxWorld) return CSVB200_ERR_INVALID_ARG;
    for (uint32_t r = 0; r < world; ++r)
        if (!all[r] || all[r]->rank != r || all[r]->world != world) return CSVB200_ERR_INVALID_ARG;
    for (uint32_t r = 0; r < world; ++r) {
        csvb200_exchange* ex = all[r];
        csvb200_ctx* ctx = ex->ctx;
        CU_TRY(ctx, cudaSetDevice(ctx->device));
        for (uint32_t q = 0; q < world; ++q) {
            const int peer_dev = all[q]->ctx->device;
            if (peer_dev != ctx->device) {
                int can = 0;
                CU_TRY(ctx, cudaDeviceCanAccessPeer(&can, ctx->device, peer_dev));
                if (!can)
                    return fail(ctx, CSVB200_ERR_EXCHANGE, "exchange: device " + std::to_string(ctx->device) +
                                                               " has no peer access to device " + std::to_string(peer_dev));
                cudaError_t e = cudaDeviceEnablePeerAccess(peer_dev, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                    cudaGetLastError();
                    return fail(ctx, CSVB200_ERR_EXCHANGE, std::string("exchange: cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
                }
                cudaGetLastError();
            }
            ex->peer[q] = all[q]->d_mbox;
        }
        int rc = upload_peer_table(ex);
        if (rc) return rc;
    }
    return CSVB200_OK;
}

void csvb200_exchange_destroy(csvb200_exchange* ex)
{
    if (!ex) return;
    cudaSetDevice(ex->ctx->device);
    cudaStreamSynchronize(ex->ctx->stream);
    for (uint32_t r = 0; r < kExMaxWorld; ++r)
        if (ex->ipc_opened[r] && ex->peer[r]) cudaIpcCloseMemHandle(ex->peer[r]);
    if (ex->d_mbox) cudaFree(ex->d_mbox);
    if (ex->d_peers) cudaFree(ex->d_peers);
    if (ex->d_row4) cudaFree(ex->d_row4);
    if (ex->h_rows) cudaFreeHost(ex->h_rows);
    cudaGetLastError();
    delete ex;
}

}  // extern "C"

namespace csvb200 {

// Host-side view of one build's slot: waits (bounded) until the rows of all ranks carry `epoch`, then runs the same
// carry chain the device runs for the lower ranks over ALL ranks.  counts[r] = true entries of rank r (rank 0 incl.
// the sentinel), carries[r] = true carry-in parity.
int exchange_wait_all(csvb200_exchange* ex, uint64_t epoch, uint64_t* counts, uint32_t* carries)
{
    csvb200_ctx* ctx = ex->ctx;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    const uint64_t* slot = ex->d_mbox + ((epoch % kExRing) * kExMaxWorld) * kExRowWords;
    const size_t bytes = (size_t)ex->world * kExRowWords * sizeof(uint64_t);
    const auto t0 = std::chrono::steady_clock::now();
    const double limit_s = std::max(10.0, 5.0 * (double)ex->timeout_ns * 1e-9);
    for (;;) {
        CU_TRY(ctx, cudaMemcpyAsync(ex->h_rows, slot, bytes, cudaMemcpyDeviceToHost, ctx->copy_stream));
        CU_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
        bool all = true, lapped = false;
        for (uint32_t r = 0; r < ex->world; ++r) {
            const uint64_t e = ex->h_rows[r * kExRowWords + 4];
            if (e != epoch) all = false;
            if (e > epoch) lapped = true;
        }
        if (all) break;
        if (lapped) return fail(ctx, CSVB200_ERR_EXCHANGE, "exchange: a rank lapped the mailbox ring (more than 1024 builds ahead)");
        if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > limit_s)
            return fail(ctx, CSVB200_ERR_EXCHANGE, "exchange: timed out waiting for the rows of all ranks");
        std::this_thread::sleep_for(std::chrono::microseconds(50));
    }
    uint64_t carry = 0;
    for (uint32_t r = 0; r < ex->world; ++r) {
        const uint64_t* row = ex->h_rows + r * kExRowWords;
        const uint64_t used = row[2] & 1ull;
        if (counts) counts[r] = (carry == used ? row[0] : row[3] - row[0]) + (r == 0 ? 1 : 0);
        if (carries) carries[r] = (uint32_t)carry;
        carry ^= (row[1] ^ row[2]) & 1ull;
    }
    return CSVB200_OK;
}

}  // namespace csvb200

extern "C" int csvb200_exchange_counts(csvb200_exchange* ex, csvb200_index* idx, uint64_t* counts, uint32_t* carries)
{
    if (!ex || !idx) return CSVB200_ERR_INVALID_ARG;
    if (idx->ex != ex) return fail(ex->ctx, CSVB200_ERR_INVALID_ARG, "index was not built through this exchange");
    int rc = csvb200_index_sync(idx);
    if (rc) return rc;
    return exchange_wait_all(ex, idx->ex_epoch, counts, carries);
}

// ---------------------------------------------------------------------------------------------------------------
// all GPUs of one process behind one call
// ---------------------------------------------------------------------------------------------------------------
struct csvb200_multi_index {
    csvb200_multi* m = nullptr;
    std::vector<csvb200_index*> seg;      // segment k on device k (global byte positions)
    std::vector<uint8_t*> d_bytes;        // device copies of the shards (kept: csvb200_index_free does not own them)
    std::vector<uint64_t> base;           // base[k] = global slot of seg[k][0]; base[G] = total length
    std::vector<size_t> cuts;             // byte shard k = global bytes [cuts[k], cuts[k + 1]), held in d_bytes[k]
    SegmentTable table{};                 // the same, as the kernels take it
    bool tape_ready = false;
    uint32_t field_cnt = 0, record_cnt = 0;
    uint64_t jump = 0;
};

struct csvb200_multi {
    std::vector<csvb200_ctx*> ctx;
    std::vector<csvb200_exchange*> ex;
    std::vector<int> device;
    bool shared_device = false;   // a device is listed twice: shards run one after another, in rank order
    std::string err;
    csvb200_multi_stats stats{};
};

namespace {

int mfail(csvb200_multi* m, int code, const std::string& msg)
{
    if (m) m->err = msg;
    return code;
}

struct ShardWork {
    int rc = CSVB200_OK;
    std::string err;
    csvb200_index* idx = nullptr;
    uint8_t* d_bytes = nullptr;
    csvb200_shard_info info{};
    double t_up = 0, t_down = 0;
};

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// phase 1 of one shard: upload, build with the exchange inside the launch, learn base / carry / count
void shard_phase1(csvb200_multi* m, int k, const uint8_t* bytes, size_t n, uint64_t goff, ShardWork* w)
{
    csvb200_ctx* ctx = m->ctx[k];
    const double t0 = now_s();
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e == cudaSuccess) e = pool_malloc((void**)&w->d_bytes, ((n + 15) & ~size_t(15)) + 16, ctx->stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        w->rc = CSVB200_ERR_OOM;
        w->err = std::string("shard input allocation: ") + cudaGetErrorString(e);
        return;
    }
    w->rc = upload(ctx, w->d_bytes, bytes, n);
    if (!w->rc) w->rc = csvb200_index_build_shard_exchange(ctx, m->ex[k], w->d_bytes, n, goff, 0, &w->idx);
    if (!w->rc) w->rc = csvb200_index_shard_info(w->idx, &w->info);
    if (w->rc) w->err = csvb200_last_error(ctx);
    w->t_up = now_s() - t0;
}

// phase 2: the segment goes straight to its place in the caller's array
void shard_phase2(csvb200_multi* m, int k, uint64_t* dst, ShardWork* w)
{
    csvb200_ctx* ctx = m->ctx[k];
    const double t0 = now_s();
    cudaSetDevice(ctx->device);
    w->rc = download(ctx, dst + w->info.base, csvb200_index_device_ptr(w->idx), (size_t)w->info.entries);
    if (w->rc) w->err = csvb200_last_error(ctx);
    w->t_down = now_s() - t0;
}

}  // namespace

extern "C" {

int csvb200_multi_create(const int* devices, int ndev, csvb200_multi** out)
{
    if (!out) return CSVB200_ERR_INVALID_ARG;
    *out = nullptr;
    if (!devices || ndev < 1 || ndev > (int)kExMaxWorld) return CSVB200_ERR_INVALID_ARG;
    csvb200_multi* m = new (std::nothrow) csvb200_multi();
    if (!m) return CSVB200_ERR_OOM;
    int rc = CSVB200_OK;
    for (int k = 0; k < ndev && !rc; ++k) {
        for (int j = 0; j < k; ++j)
            if (devices[j] == devices[k]) m->shared_device = true;
        csvb200_ctx* c = nullptr;
        rc = csvb200_ctx_create(devices[k], &c);
        if (rc) break;
        c->io_threads = std::max(2, default_io_threads() / ndev);   // the host's copy threads are shared by all devices
        m->ctx.push_back(c);
        m->device.push_back(devices[k]);
        csvb200_exchange* ex = nullptr;
        rc = csvb200_exchange_create(c, (uint32_t)k, (uint32_t)ndev, &ex);
        if (rc) break;
        m->ex.push_back(ex);
    }
    if (!rc && ndev > 1) rc = csvb200_exchange_connect_local(m->ex.data(), (uint32_t)ndev);
    // index segments come from each device's stream-ordered pool: grant every other listed device access to it, so a
    // lookup kernel on device j can read a segment that lives on device k (csvb200_multi_seek_fields)
    for (int k = 0; k < ndev && !rc; ++k) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, devices[k]) != cudaSuccess) {
            cudaGetLastError();
            continue;
        }
        std::vector<cudaMemAccessDesc> desc;
        for (int j = 0; j < ndev; ++j) {
            if (devices[j] == devices[k]) continue;
            bool seen = false;
            for (const cudaMemAccessDesc& d : desc) seen = seen || d.location.id == devices[j];
            if (seen) continue;
            cudaMemAccessDesc d{};
            d.location.type = cudaMemLocationTypeDevice;
            d.location.id = devices[j];
            d.flags = cudaMemAccessFlagsProtReadWrite;
            desc.push_back(d);
        }
        if (!desc.empty() && cudaMemPoolSetAccess(pool, desc.data(), desc.size()) != cudaSuccess) {
            cudaGetLastError();
            rc = CSVB200_ERR_EXCHANGE;
        }
    }
    if (rc) {
        csvb200_multi_destroy(m);
        return rc;
    }
    *out = m;
    return CSVB200_OK;
}

void csvb200_multi_destroy(csvb200_multi* m)
{
    if (!m) return;
    for (csvb200_exchange* ex : m->ex) csvb200_exchange_destroy(ex);
    for (csvb200_ctx* c : m->ctx) csvb200_ctx_destroy(c);
    delete m;
}

const char* csvb200_multi_last_error(const csvb200_multi* m) { return m ? m->err.c_str() : "null multi"; }

int csvb200_multi_device_count(const csvb200_multi* m) { return m ? (int)m->ctx.size() : 0; }

int csvb200_multi_last_stats(const csvb200_multi* m, csvb200_multi_stats* out)
{
    if (!m || !out) return CSVB200_ERR_INVALID_ARG;
    *out = m->stats;
    return CSVB200_OK;
}

}  // extern "C"

namespace {

int make_cuts(csvb200_multi* m, size_t n, const size_t* cuts_in, std::vector<size_t>& cuts)
{
    const int G = (int)m->ctx.size();
    cuts.resize(G + 1);
    for (int k = 0; k <= G; ++k) {
        if (cuts_in) {
            cuts[k] = cuts_in[k];
        } else {
            // deliberately not record-, 16- or 64-byte aligned (SURVEY 8d config 4): correctness never depends on the cuts
            cuts[k] = k == 0 ? 0 : k == G ? n : std::min(n, (size_t)((unsigned __int128)n * k / G) + 37u * k + 13u);
        }
        if (k > 0 && cuts[k] < cuts[k - 1]) return mfail(m, CSVB200_ERR_INVALID_ARG, "cuts must be non-decreasing");
    }
    if (cuts[0] != 0 || cuts[G] != n) return mfail(m, CSVB200_ERR_INVALID_ARG, "cuts must span [0, n]");
    return CSVB200_OK;
}

template <class F>
void run_phase(csvb200_multi* m, F&& fn)
{
    const int G = (int)m->ctx.size();
    if (m->shared_device || G == 1) {
        for (int k = 0; k < G; ++k) fn(k);   // rank order: a rank only ever waits for lower ranks
    } else {
        std::vector<std::thread> th;
        for (int k = 0; k < G; ++k) th.emplace_back(fn, k);
        for (std::thread& t : th) t.join();
    }
}

}  // namespace

extern "C" {

int csvb200_multi_index_build(csvb200_multi* m, const uint8_t* host_bytes, size_t n, const size_t* cuts_in,
                              csvb200_multi_index** out)
{
    if (!m || !out || (n && !host_bytes)) return mfail(m, CSVB200_ERR_INVALID_ARG, "null argument");
    *out = nullptr;
    const int G = (int)m->ctx.size();
    std::vector<size_t> cuts;
    int rc = make_cuts(m, n, cuts_in, cuts);
    if (rc) return rc;
    std::vector<ShardWork> work(G);
    run_phase(m, [&](int k) { shard_phase1(m, k, host_bytes + cuts[k], cuts[k + 1] - cuts[k], cuts[k], &work[k]); });
    for (int k = 0; k < G && !rc; ++k)
        if (work[k].rc) rc = mfail(m, work[k].rc, "shard " + std::to_string(k) + ": " + work[k].err);
    csvb200_multi_index* mi = rc ? nullptr : new (std::nothrow) csvb200_multi_index();
    if (!rc && !mi) rc = mfail(m, CSVB200_ERR_OOM, "host allocation failed");
    if (rc) {
        for (int k = 0; k < G; ++k) {
            cudaSetDevice(m->ctx[k]->device);
            if (work[k].idx) csvb200_index_free(work[k].idx);
            if (work[k].d_bytes) cudaFreeAsync(work[k].d_bytes, m->ctx[k]->stream);
        }
        cudaGetLastError();
        return rc;
    }
    mi->m = m;
    mi->cuts = cuts;
    mi->table.nseg = (uint32_t)G;
    for (int k = 0; k < G; ++k) {
        mi->seg.push_back(work[k].idx);
        mi->d_bytes.push_back(work[k].d_bytes);
        mi->base.push_back(work[k].info.base);
        mi->table.ptr[k] = csvb200_index_device_ptr(work[k].idx);
        mi->table.base[k] = work[k].info.base;
    }
    mi->base.push_back(work[G - 1].info.base + work[G - 1].info.entries);
    mi->table.base[G] = mi->base[G];
    *out = mi;
    return CSVB200_OK;
}

void csvb200_multi_index_free(csvb200_multi_index* mi)
{
    if (!mi) return;
    for (size_t k = 0; k < mi->seg.size(); ++k) {
        csvb200_ctx* ctx = mi->m->ctx[k];
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        if (mi->seg[k]) csvb200_index_free(mi->seg[k]);
        if (mi->d_bytes[k]) cudaFreeAsync(mi->d_bytes[k], ctx->stream);
    }
    cudaGetLastError();
    delete mi;
}

size_t csvb200_multi_index_len(const csvb200_multi_index* mi) { return mi ? (size_t)mi->base.back() : 0; }

int csvb200_multi_index_segment(const csvb200_multi_index* mi, int k, uint64_t* base, uint64_t* entries, int* device)
{
    if (!mi || k < 0 || k >= (int)mi->seg.size()) return CSVB200_ERR_INVALID_ARG;
    if (base) *base = mi->base[k];
    if (entries) *entries = mi->base[k + 1] - mi->base[k];
    if (device) *device = mi->m->ctx[k]->device;
    return CSVB200_OK;
}

int csvb200_multi_index_copy_out(csvb200_multi_index* mi, uint64_t* dst, size_t dst_cap)
{
    if (!mi || !dst) return CSVB200_ERR_INVALID_ARG;
    csvb200_multi* m = mi->m;
    if (mi->base.back() > dst_cap) return mfail(m, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    const int G = (int)mi->seg.size();
    std::vector<int> rcs(G, 0);
    run_phase(m, [&](int k) {
        rcs[k] = download(m->ctx[k], dst + mi->base[k], mi->table.ptr[k], (size_t)(mi->base[k + 1] - mi->base[k]));
    });
    for (int k = 0; k < G; ++k)
        if (rcs[k]) return mfail(m, rcs[k], "segment " + std::to_string(k) + ": " + csvb200_last_error(m->ctx[k]));
    return CSVB200_OK;
}

int csvb200_multi_tape_init(csvb200_multi_index* mi, uint32_t field_cnt, int crlf, uint32_t* record_cnt, uint64_t* jump)
{
    if (!mi) return CSVB200_ERR_INVALID_ARG;
    const uint64_t len = mi->base.back();
    const uint64_t j = crlf ? (uint64_t)field_cnt + 1 : (uint64_t)field_cnt;   // src/tape.rs:318-321
    if (j == 0 || len == 0) return mfail(mi->m, CSVB200_ERR_INVALID_ARG, "field_cnt must be >= 1");
    mi->field_cnt = field_cnt;
    mi->jump = j;
    mi->record_cnt = (uint32_t)((len - 1) / j);                                 // src/tape.rs:323-325
    mi->tape_ready = true;
    if (record_cnt) *record_cnt = mi->record_cnt;
    if (jump) *jump = j;
    if ((len - 1) % j != 0)                                                     // src/tape.rs:327,342-344
        return mfail(mi->m, CSVB200_ERR_INVALID_CSV_FORMAT, csvb200_status_string(CSVB200_ERR_INVALID_CSV_FORMAT));
    return CSVB200_OK;
}

// queries [q0, q1) on device k: host arrays in / out
static int seek_share(csvb200_multi_index* mi, int k, const uint32_t* rec, const uint32_t* fld, size_t q0, size_t q1,
                      csvb200_range* out, uint32_t* oob_out)
{
    csvb200_ctx* ctx = mi->m->ctx[k];
    const size_t nq = q1 - q0;
    if (nq == 0) return CSVB200_OK;
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    DevBuf d_rec, d_fld, d_out, d_oob;
    CU_TRY(ctx, d_rec.alloc(nq * sizeof(uint32_t), ctx->stream));
    if (fld) CU_TRY(ctx, d_fld.alloc(nq * sizeof(uint32_t), ctx->stream));
    CU_TRY(ctx, d_out.alloc(nq * sizeof(csvb200_range), ctx->stream));
    CU_TRY(ctx, d_oob.alloc(sizeof(uint32_t), ctx->stream));
    CU_TRY(ctx, cudaMemsetAsync(d_oob.p, 0, sizeof(uint32_t), ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(d_rec.p, rec + q0, nq * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    if (fld) CU_TRY(ctx, cudaMemcpyAsync(d_fld.p, fld + q0, nq * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    LookupParams p{};
    p.index_len = mi->base.back();
    p.record_cnt = mi->record_cnt;
    p.field_cnt = mi->field_cnt;
    p.row_size = (uint32_t)mi->jump;
    p.rec = d_rec.as<uint32_t>();
    p.fld = fld ? d_fld.as<uint32_t>() : nullptr;
    p.nq = nq;
    p.ranges = d_out.as<uint64_t>();
    p.oob = d_oob.as<uint32_t>();
    CU_TRY(ctx, launch_seek_sharded(p, mi->table, ctx->stream));
    ctx->launches += 1;
    CU_TRY(ctx, cudaMemcpyAsync(out + q0, d_out.p, nq * sizeof(csvb200_range), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(oob_out, d_oob.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return CSVB200_OK;
}

static int multi_seek(csvb200_multi_index* mi, const uint32_t* rec, const uint32_t* fld, size_t nq, csvb200_range* out)
{
    if (!mi) return CSVB200_ERR_INVALID_ARG;
    csvb200_multi* m = mi->m;
    if (!mi->tape_ready) return mfail(m, CSVB200_ERR_INVALID_STATE, "csvb200_multi_tape_init has not been called");
    if (nq == 0) return CSVB200_OK;
    if (!rec || !out) return mfail(m, CSVB200_ERR_INVALID_ARG, "null argument");
    // every device resolves an equal share of the batch; a slot owned by another GPU is one NVLink read
    const int G = (int)mi->seg.size();
    std::vector<int> rcs(G, 0);
    std::vector<uint32_t> oob(G, 0);
    run_phase(m, [&](int k) {
        const size_t q0 = nq * k / G, q1 = nq * (k + 1) / G;
        rcs[k] = seek_share(mi, k, rec, fld, q0, q1, out, &oob[k]);
    });
    for (int k = 0; k < G; ++k) {
        if (rcs[k]) return mfail(m, rcs[k], "device " + std::to_string(k) + ": " + csvb200_last_error(m->ctx[k]));
        if (oob[k]) return mfail(m, CSVB200_ERR_OUT_OF_BOUNDS, "lookup slot past the end of the index");
    }
    return CSVB200_OK;
}

int csvb200_multi_seek_fields(csvb200_multi_index* mi, const uint32_t* rec, const uint32_t* fld, size_t nq, csvb200_range* out)
{
    if (mi && nq && !fld) return mfail(mi->m, CSVB200_ERR_INVALID_ARG, "null argument");
    return multi_seek(mi, rec, fld, nq, out);
}

int csvb200_multi_seek_records(csvb200_multi_index* mi, const uint32_t* rec, size_t nq, csvb200_range* out)
{
    return multi_seek(mi, rec, nullptr, nq, out);
}

// device arrays that live on device k in / out; asynchronous on that device's context stream (benchmarks)
int csvb200_multi_seek_fields_device(csvb200_multi_index* mi, int k, const uint32_t* d_rec, const uint32_t* d_fld, size_t nq,
                                     csvb200_range* d_out)
{
    if (!mi || k < 0 || k >= (int)mi->seg.size()) return CSVB200_ERR_INVALID_ARG;
    csvb200_ctx* ctx = mi->m->ctx[k];
    if (!mi->tape_ready) return mfail(mi->m, CSVB200_ERR_INVALID_STATE, "csvb200_multi_tape_init has not been called");
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    LookupParams p{};
    p.index_len = mi->base.back();
    p.record_cnt = mi->record_cnt;
    p.field_cnt = mi->field_cnt;
    p.row_size = (uint32_t)mi->jump;
    p.rec = d_rec;
    p.fld = d_fld;
    p.nq = nq;
    p.ranges = reinterpret_cast<uint64_t*>(d_out);
    p.oob = reinterpret_cast<uint32_t*>(ctx->d_cells + (kCells - 1) * kCellWords);
    CU_TRY(ctx, launch_seek_sharded(p, mi->table, ctx->stream));
    ctx->launches += 1;
    return CSVB200_OK;
}

void* csvb200_multi_stream(csvb200_multi* m, int k)
{
    return (m && k >= 0 && k < (int)m->ctx.size()) ? (void*)m->ctx[k]->stream : nullptr;
}

int csvb200_multi_index_build_to_host(csvb200_multi* m, const uint8_t* host_bytes, size_t n, const size_t* cuts_in,
                                      uint64_t* dst, size_t dst_cap, size_t* len_out)
{
    if (!m || !len_out || (n && !host_bytes)) return mfail(m, CSVB200_ERR_INVALID_ARG, "null argument");
    const int G = (int)m->ctx.size();
    std::vector<size_t> cuts;
    {
        int rc0 = make_cuts(m, n, cuts_in, cuts);
        if (rc0) return rc0;
    }
    const double t0 = now_s();
    std::vector<ShardWork> work(G);
    auto first_error = [&]() -> int {
        for (int k = 0; k < G; ++k)
            if (work[k].rc) return mfail(m, work[k].rc, "shard " + std::to_string(k) + ": " + work[k].err);
        return CSVB200_OK;
    };
    auto cleanup = [&]() {
        for (int k = 0; k < G; ++k) {
            cudaSetDevice(m->ctx[k]->device);
            if (work[k].idx) csvb200_index_free(work[k].idx);
            if (work[k].d_bytes) cudaFreeAsync(work[k].d_bytes, m->ctx[k]->stream);
        }
        cudaGetLastError();
    };
    run_phase(m, [&](int k) { shard_phase1(m, k, host_bytes + cuts[k], cuts[k + 1] - cuts[k], cuts[k], &work[k]); });
    int rc = first_error();
    size_t total = 0;
    if (!rc) {
        total = (size_t)(work[G - 1].info.base + work[G - 1].info.entries);
        *len_out = total;
        if (total > dst_cap || (total && !dst)) rc = mfail(m, CSVB200_ERR_CAPACITY, "destination index buffer too small");
    }
    if (!rc) {
        run_phase(m, [&](int k) { shard_phase2(m, k, dst, &work[k]); });
        rc = first_error();
    }
    m->stats = csvb200_multi_stats{};
    for (int k = 0; k < G; ++k) {
        m->stats.upload_seconds = std::max(m->stats.upload_seconds, work[k].t_up);
        m->stats.download_seconds = std::max(m->stats.download_seconds, work[k].t_down);
        if (work[k].info.redone) m->stats.redone_mask |= 1u << k;
        if (work[k].info.carry_in) m->stats.carry_mask |= 1u << k;
    }
    m->stats.entries = total;
    cleanup();
    m->stats.seconds = now_s() - t0;
    return rc;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// the values behind a batch of lookups over the distributed index: every device resolves a share of the batch, reading
// index slots and bytes from whichever device holds them (peer loads into the shards, nothing is staged)
// ---------------------------------------------------------------------------------------------------------------
namespace {

int first_device_error(csvb200_multi* m, const std::vector<int>& rcs);

ShardBytes shard_bytes(const csvb200_multi_index* mi)
{
    ShardBytes sb{};
    sb.nshard = (uint32_t)mi->seg.size();
    for (size_t k = 0; k < mi->seg.size(); ++k) sb.ptr[k] = mi->d_bytes[k];
    for (size_t k = 0; k < mi->cuts.size(); ++k) sb.cut[k] = mi->cuts[k];
    return sb;
}

ValuesParams multi_values_params(const csvb200_multi_index* mi, const uint32_t* rec, const uint32_t* fld, size_t nq,
                                 uint32_t flags)
{
    ValuesParams p{};
    p.index_len = mi->base.back();
    p.record_cnt = mi->record_cnt;
    p.field_cnt = mi->field_cnt;
    p.row_size = (uint32_t)mi->jump;
    p.flags = flags;
    p.rec = rec;
    p.fld = fld;
    p.nq = nq;
    return p;
}

int multi_values_args(csvb200_multi_index* mi, const void* rec, const void* fld, size_t nq, uint32_t flags, const void* offsets)
{
    csvb200_multi* m = mi->m;
    if (!mi->tape_ready) return mfail(m, CSVB200_ERR_INVALID_STATE, "csvb200_multi_tape_init has not been called");
    if (!offsets || (nq && !rec)) return mfail(m, CSVB200_ERR_INVALID_ARG, "null argument");
    if (flags & ~(CSVB200_FIELD_UNQUOTE | CSVB200_FIELD_TRIM)) return mfail(m, CSVB200_ERR_INVALID_ARG, "unknown field flags");
    if (flags && !fld) return mfail(m, CSVB200_ERR_INVALID_ARG, "flags apply to fields only (fld == NULL: records)");
    return CSVB200_OK;
}

// one device's share of a batch: queries [q0, q1) and what its device made of them
struct ValuesShare {
    size_t q0 = 0, q1 = 0;
    DevBuf rec, fld, off, found, cnt, out;
    uint64_t total = 0, start = 0;
    uint32_t counts[2] = {0, 0};
};

}  // namespace

extern "C" int csvb200_multi_seek_values(csvb200_multi_index* mi, const uint32_t* rec, const uint32_t* fld, size_t nq,
                                         uint32_t flags, uint64_t* out_offsets, uint8_t* out, size_t out_cap, size_t* out_len,
                                         uint64_t* found_bits)
{
    if (!mi) return CSVB200_ERR_INVALID_ARG;
    csvb200_multi* m = mi->m;
    int rc = multi_values_args(mi, rec, fld, nq, flags, out_offsets);
    if (rc) return rc;
    if (!out_len) return mfail(m, CSVB200_ERR_INVALID_ARG, "null argument");
    *out_len = 0;
    out_offsets[0] = 0;
    if (nq == 0) return CSVB200_OK;
    // one share per device, as multi_seek splits a batch; the boundaries are multiples of 64 queries, so that every
    // device writes whole words of the found bits
    const int G = (int)mi->seg.size();
    std::vector<ValuesShare> sh(G);
    for (int k = 0; k < G; ++k) {
        sh[k].q0 = k == 0 ? 0 : sh[k - 1].q1;
        sh[k].q1 = k + 1 == G ? nq : std::max(sh[k].q0, std::min(nq, (nq * (k + 1) / G + 63) / 64 * 64));
    }
    const ShardBytes sb = shard_bytes(mi);
    std::vector<int> rcs(G, CSVB200_OK);
    // pass 1: lengths, offsets from 0 and found bits of every share on its device; only the totals come back
    run_phase(m, [&](int k) {
        csvb200_ctx* ctx = m->ctx[k];
        ValuesShare& s = sh[k];
        const size_t n = s.q1 - s.q0;
        if (n == 0) return;
        rcs[k] = [&]() -> int {
            CU_TRY(ctx, cudaSetDevice(ctx->device));
            CU_TRY(ctx, s.rec.alloc(n * sizeof(uint32_t), ctx->stream));
            if (fld) CU_TRY(ctx, s.fld.alloc(n * sizeof(uint32_t), ctx->stream));
            CU_TRY(ctx, s.off.alloc((n + 1) * sizeof(uint64_t), ctx->stream));
            if (found_bits) CU_TRY(ctx, s.found.alloc((n + 63) / 64 * sizeof(uint64_t), ctx->stream));
            CU_TRY(ctx, s.cnt.alloc(2 * sizeof(uint32_t), ctx->stream));
            CU_TRY(ctx, cudaMemsetAsync(s.cnt.p, 0, 2 * sizeof(uint32_t), ctx->stream));
            CU_TRY(ctx, cudaMemcpyAsync(s.rec.p, rec + s.q0, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
            if (fld) CU_TRY(ctx, cudaMemcpyAsync(s.fld.p, fld + s.q0, n * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
            ValuesParams p = multi_values_params(mi, s.rec.as<uint32_t>(), fld ? s.fld.as<uint32_t>() : nullptr, n, flags);
            p.offsets = s.off.as<uint64_t>();
            p.found = found_bits ? s.found.as<uint32_t>() : nullptr;
            p.counts = s.cnt.as<uint32_t>();
            int rc2 = values_enqueue(ctx, p, nullptr, &mi->table, &sb, false);
            if (rc2) return rc2;
            CU_TRY(ctx, cudaMemcpyAsync(&s.total, s.off.as<uint64_t>() + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaMemcpyAsync(s.counts, s.cnt.p, sizeof(s.counts), cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            return CSVB200_OK;
        }();
    });
    rc = first_device_error(m, rcs);
    uint64_t total = 0;
    bool oob = false, outside = false;
    for (ValuesShare& s : sh) {
        s.start = total;
        total += s.total;
        oob = oob || s.counts[0];
        outside = outside || s.counts[1];
    }
    if (!rc && oob) rc = mfail(m, CSVB200_ERR_OUT_OF_BOUNDS, "lookup slot past the end of the index");
    if (!rc && outside) rc = mfail(m, CSVB200_ERR_OUT_OF_BOUNDS, "value lies outside the input");
    const bool small = total > out_cap, write = !small && out != nullptr;
    if (!rc) {
        *out_len = (size_t)total;
        // pass 2: the values (when they fit), the offsets again with the share's start added, and the found bits go
        // from every device straight to their place in the caller's arrays; the offsets come down even when the values
        // do not (CSVB200_ERR_CAPACITY, the sizing call)
        run_phase(m, [&](int k) {
            csvb200_ctx* ctx = m->ctx[k];
            ValuesShare& s = sh[k];
            const size_t n = s.q1 - s.q0;
            if (n == 0) return;
            rcs[k] = [&]() -> int {
                CU_TRY(ctx, cudaSetDevice(ctx->device));
                ValuesParams p = multi_values_params(mi, s.rec.as<uint32_t>(), fld ? s.fld.as<uint32_t>() : nullptr, n, flags);
                p.offsets = s.off.as<uint64_t>();
                if (write && s.total) {
                    CU_TRY(ctx, s.out.alloc(s.total, ctx->stream));
                    p.out = s.out.as<uint8_t>();
                    p.out_cap = s.total;
                    CU_TRY(ctx, launch_values_write_sharded(p, mi->table, sb, ctx->stream));
                    ctx->launches += 1;
                }
                p.out = nullptr;
                p.offset_base = s.start;
                p.counts = s.cnt.as<uint32_t>();
                int rc2 = values_enqueue(ctx, p, nullptr, &mi->table, &sb, false);
                if (rc2) return rc2;
                // adjacent shares share one offset: each brings its own queries' offsets, the last share the end too
                const size_t n_off = n + (s.q1 == nq ? 1 : 0);
                CU_TRY(ctx, cudaMemcpyAsync(out_offsets + s.q0, s.off.p, n_off * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
                if (found_bits)
                    CU_TRY(ctx, cudaMemcpyAsync(found_bits + s.q0 / 64, s.found.p, (n + 63) / 64 * sizeof(uint64_t),
                                                cudaMemcpyDeviceToHost, ctx->stream));
                if (write && s.total)
                    CU_TRY(ctx, cudaMemcpyAsync(out + s.start, s.out.p, s.total, cudaMemcpyDeviceToHost, ctx->stream));
                CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
                return CSVB200_OK;
            }();
        });
        rc = first_device_error(m, rcs);
    }
    // every buffer goes back to the pool of the device it came from, on that device's stream
    run_phase(m, [&](int k) {
        cudaSetDevice(m->ctx[k]->device);
        ValuesShare& s = sh[k];
        s.rec.reset();
        s.fld.reset();
        s.off.reset();
        s.found.reset();
        s.cnt.reset();
        s.out.reset();
    });
    cudaGetLastError();
    if (rc) return rc;
    if (small) return mfail(m, CSVB200_ERR_CAPACITY, "values destination too small");
    if (total && !out) return mfail(m, CSVB200_ERR_INVALID_ARG, "null argument");
    return CSVB200_OK;
}

extern "C" int csvb200_multi_seek_values_device(csvb200_multi_index* mi, int k, const uint32_t* d_rec, const uint32_t* d_fld,
                                                size_t nq, uint32_t flags, uint64_t* d_offsets, uint8_t* d_out, size_t out_cap,
                                                uint64_t* d_found_bits)
{
    if (!mi || k < 0 || k >= (int)mi->seg.size()) return CSVB200_ERR_INVALID_ARG;
    int rc = multi_values_args(mi, d_rec, d_fld, nq, flags, d_offsets);
    if (rc) return rc;
    csvb200_ctx* ctx = mi->m->ctx[k];
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    ValuesParams p = multi_values_params(mi, d_rec, d_fld, nq, flags);
    p.offsets = d_offsets;
    p.out = d_out;
    p.out_cap = out_cap;
    p.found = reinterpret_cast<uint32_t*>(d_found_bits);
    // out-of-bounds slots are reported as None on this asynchronous path
    p.counts = reinterpret_cast<uint32_t*>(ctx->d_cells + (kCells - 1) * kCellWords);
    const ShardBytes sb = shard_bytes(mi);
    return values_enqueue(ctx, p, nullptr, &mi->table, &sb, true);
}

// ---------------------------------------------------------------------------------------------------------------
// column materialisation over the distributed index: every device materialises the records whose bytes it holds
// ---------------------------------------------------------------------------------------------------------------
namespace {

// An index pointer to hand the kernels so that index[s] addresses global slot s, given the array that starts at slot
// first_slot.  The pointer itself points before the array; that is safe because the kernels read index[s] only for the
// slots of the records they are given, and a piece is only given records whose slots all lie in [first_slot, end).
const uint64_t* by_global_slot(const uint64_t* first, uint64_t first_slot)
{
    return reinterpret_cast<const uint64_t*>(reinterpret_cast<uintptr_t>(first) - first_slot * sizeof(uint64_t));
}

// one piece of a request (record_split.h) and what its device made of it
struct MatPiece {
    RecordPiece r{};
    uint64_t pos = 0;             // window position of its first record
    int k = 0;                    // the device that runs it
    MatSource src{};
    DevBuf row_slots, row_bytes;  // boundary record: its index slots and byte span, staged on device k
    DevBuf d_off[kMatMaxCols], d_out[kMatMaxCols];
    uint64_t total[kMatMaxCols] = {}, start[kMatMaxCols] = {};
};

// Copies the slots and the byte span of boundary record p->r.first to device p->k, from whichever devices hold them.
int stage_boundary_row(csvb200_multi_index* mi, MatPiece* p)
{
    csvb200_ctx* ctx = mi->m->ctx[p->k];
    const int dev = ctx->device;
    const uint64_t lo = (uint64_t)(uint32_t)(p->r.first + 1u) * mi->jump, hi = lo + mi->jump;
    CU_TRY(ctx, p->row_slots.alloc((hi - lo + 1) * sizeof(uint64_t), ctx->stream));
    uint64_t* slots = p->row_slots.as<uint64_t>();
    for (uint32_t j = p->r.seg_lo; j <= p->r.seg_hi; ++j) {
        const uint64_t a = std::max(lo, mi->base[j]), b = std::min(hi + 1, mi->base[j + 1]);
        if (a < b)
            CU_TRY(ctx, cudaMemcpyPeerAsync(slots + (a - lo), dev, mi->table.ptr[j] + (a - mi->base[j]), mi->m->ctx[j]->device,
                                            (b - a) * sizeof(uint64_t), ctx->stream));
    }
    uint64_t ends[2];
    CU_TRY(ctx, cudaMemcpyAsync(&ends[0], slots, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaMemcpyAsync(&ends[1], slots + (hi - lo), sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    // every value of the row lies in (index[lo], index[hi]); the staged bytes start at index[lo] itself, so no position
    // the kernels compute from the row's slots falls below the span
    const uint64_t p0 = ends[0], p1 = std::max(ends[0], ends[1]);
    CU_TRY(ctx, p->row_bytes.alloc(((p1 - p0 + 15) & ~uint64_t(15)) + 16, ctx->stream));
    for (size_t j = 0; j + 1 < mi->cuts.size(); ++j) {
        const uint64_t a = std::max<uint64_t>(p0, mi->cuts[j]), b = std::min<uint64_t>(p1, mi->cuts[j + 1]);
        if (a < b)
            CU_TRY(ctx, cudaMemcpyPeerAsync(p->row_bytes.as<uint8_t>() + (a - p0), dev, mi->d_bytes[j] + (a - mi->cuts[j]),
                                            mi->m->ctx[j]->device, b - a, ctx->stream));
    }
    p->src.index = by_global_slot(slots, lo);
    p->src.index_len = hi + 1;
    p->src.bytes = p->row_bytes.as<uint8_t>();
    p->src.n = p1 - p0;
    p->src.pos_bias = p0;
    return CSVB200_OK;
}

}  // namespace

extern "C" int csvb200_multi_materialize_columns(csvb200_multi_index* mi, const uint32_t* fields, uint32_t ncols,
                                                 uint32_t first_record, uint32_t nrec, uint32_t flags,
                                                 uint64_t* const* out_offsets, uint8_t* const* outs, const size_t* out_caps,
                                                 size_t* out_lens)
{
    if (!mi) return CSVB200_ERR_INVALID_ARG;
    csvb200_multi* m = mi->m;
    if (!mi->tape_ready) return mfail(m, CSVB200_ERR_INVALID_STATE, "csvb200_multi_tape_init has not been called");
    if (flags & ~(CSVB200_FIELD_UNQUOTE | CSVB200_FIELD_TRIM)) return mfail(m, CSVB200_ERR_INVALID_ARG, "unknown field flags");
    if (!fields || !out_offsets || !out_lens || ncols == 0 || ncols > kMatMaxCols)
        return mfail(m, CSVB200_ERR_INVALID_ARG, "1 <= ncols <= 32 and non-null arrays");
    for (uint32_t c = 0; c < ncols; ++c)
        if (!out_offsets[c]) return mfail(m, CSVB200_ERR_INVALID_ARG, "null argument");
    // the kernels compute slots in u32, as the reference does; past 2^32 slots that would address the wrong segment
    if (mi->base.back() > (1ull << 32)) return mfail(m, CSVB200_ERR_INVALID_ARG, "index of more than 2^32 entries");
    const int G = (int)mi->seg.size();
    const std::vector<RecordPiece> split =
        split_records(mi->base.data(), (uint32_t)G, mi->jump, mi->record_cnt, first_record, nrec);
    std::vector<MatPiece> pieces(split.size());
    for (size_t i = 0, pos = 0; i < split.size(); pos += split[i].count, ++i) {
        MatPiece& p = pieces[i];
        p.r = split[i];
        p.pos = pos;
        // interior records read segment k and shard k in place; dead records read nothing, any device will do
        p.k = p.r.seg_lo < (uint32_t)G ? (int)p.r.seg_lo : G - 1;
        p.src = MatSource{by_global_slot(mi->table.ptr[p.k], mi->base[p.k]), mi->base[p.k + 1], mi->d_bytes[p.k],
                          mi->cuts[p.k + 1] - mi->cuts[p.k], mi->cuts[p.k], mi->record_cnt, mi->field_cnt, (uint32_t)mi->jump};
    }
    std::vector<int> rcs(G, CSVB200_OK);
    auto first_error = [&]() -> int {
        for (int k = 0; k < G; ++k)
            if (rcs[k]) return mfail(m, rcs[k], "device " + std::to_string(k) + ": " + csvb200_last_error(m->ctx[k]));
        return CSVB200_OK;
    };
    // offsets pass: every piece's value lengths, scanned on its device; only the column totals come back
    run_phase(m, [&](int k) {
        csvb200_ctx* ctx = m->ctx[k];
        rcs[k] = [&]() -> int {
            CU_TRY(ctx, cudaSetDevice(ctx->device));
            for (MatPiece& p : pieces) {
                if (p.k != k) continue;
                if (!p.r.interior() && p.r.seg_lo < (uint32_t)G) {
                    int rc = stage_boundary_row(mi, &p);
                    if (rc) return rc;
                }
                uint64_t* d_off[kMatMaxCols];
                for (uint32_t c = 0; c < ncols; ++c) {
                    CU_TRY(ctx, p.d_off[c].alloc(((size_t)p.r.count + 1) * sizeof(uint64_t), ctx->stream));
                    d_off[c] = p.d_off[c].as<uint64_t>();
                }
                int rc = materialize_multi_enqueue(ctx, p.src, fields, ncols, p.r.first, p.r.count, flags, d_off, nullptr,
                                                   nullptr, nullptr, true, false);
                if (rc) return rc;
                for (uint32_t c = 0; c < ncols; ++c)
                    CU_TRY(ctx, cudaMemcpyAsync(&p.total[c], d_off[c] + p.r.count, sizeof(uint64_t), cudaMemcpyDeviceToHost,
                                                ctx->stream));
            }
            CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            return CSVB200_OK;
        }();
    });
    int rc = first_error();
    bool small = false, any = false, write = false;
    if (!rc) {
        for (uint32_t c = 0; c < ncols; ++c) {
            uint64_t at = 0;
            for (MatPiece& p : pieces) {
                p.start[c] = at;
                at += p.total[c];
            }
            out_lens[c] = (size_t)at;
            if (at > (out_caps ? out_caps[c] : 0)) small = true;
            if (at) any = true;
        }
        write = !small && any && outs;
        for (uint32_t c = 0; write && c < ncols; ++c)
            if (out_lens[c] && !outs[c]) write = false;
        if (nrec == 0)
            for (uint32_t c = 0; c < ncols; ++c) out_offsets[c][0] = 0;
        // write pass: values into device buffers by the offsets of the first pass, then the offsets pass again with
        // every column's start added, and both straight to their place in the caller's arrays.  The offsets come down
        // even when the values do not (CSVB200_ERR_CAPACITY, the sizing call).
        run_phase(m, [&](int k) {
            csvb200_ctx* ctx = m->ctx[k];
            rcs[k] = [&]() -> int {
                CU_TRY(ctx, cudaSetDevice(ctx->device));
                for (size_t i = 0; i < pieces.size(); ++i) {
                    MatPiece& p = pieces[i];
                    if (p.k != k) continue;
                    uint64_t* d_off[kMatMaxCols];
                    uint8_t* d_out[kMatMaxCols];
                    size_t caps[kMatMaxCols];
                    bool values = false;
                    for (uint32_t c = 0; c < ncols; ++c) {
                        d_off[c] = p.d_off[c].as<uint64_t>();
                        d_out[c] = nullptr;
                        caps[c] = write ? (size_t)p.total[c] : 0;
                        if (caps[c]) {
                            CU_TRY(ctx, p.d_out[c].alloc(caps[c], ctx->stream));
                            d_out[c] = p.d_out[c].as<uint8_t>();
                            values = true;
                        }
                    }
                    int rc = CSVB200_OK;
                    if (values)
                        rc = materialize_multi_enqueue(ctx, p.src, fields, ncols, p.r.first, p.r.count, flags, d_off, d_out,
                                                       caps, nullptr, false, true);
                    if (!rc)
                        rc = materialize_multi_enqueue(ctx, p.src, fields, ncols, p.r.first, p.r.count, flags, d_off, nullptr,
                                                       nullptr, p.start, true, false);
                    if (rc) return rc;
                    // adjacent pieces share one offset: each brings its own records' offsets, the last piece the end too
                    const size_t n_off = (size_t)p.r.count + (i + 1 == pieces.size() ? 1 : 0);
                    for (uint32_t c = 0; c < ncols; ++c) {
                        CU_TRY(ctx, cudaMemcpyAsync(out_offsets[c] + p.pos, d_off[c], n_off * sizeof(uint64_t),
                                                    cudaMemcpyDeviceToHost, ctx->stream));
                        if (caps[c])
                            CU_TRY(ctx, cudaMemcpyAsync(outs[c] + p.start[c], d_out[c], caps[c], cudaMemcpyDeviceToHost,
                                                        ctx->stream));
                    }
                }
                CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
                return CSVB200_OK;
            }();
        });
        rc = first_error();
    }
    // every buffer goes back to the pool of the device it came from, on that device's stream
    run_phase(m, [&](int k) {
        cudaSetDevice(m->ctx[k]->device);
        for (MatPiece& p : pieces) {
            if (p.k != k) continue;
            p.row_slots.reset();
            p.row_bytes.reset();
            for (uint32_t c = 0; c < ncols; ++c) {
                p.d_off[c].reset();
                p.d_out[c].reset();
            }
        }
    });
    cudaGetLastError();
    if (rc) return rc;
    if (small) return mfail(m, CSVB200_ERR_CAPACITY, "materialize destination too small");
    if (!any) return CSVB200_OK;
    if (!write) return mfail(m, CSVB200_ERR_INVALID_ARG, "null argument");
    return CSVB200_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// tape validation, UTF-8 validation and chunks over the distributed index: every device checks its own segment and
// shard in place with the one-GPU kernels, and the host joins the answers across the cuts
// ---------------------------------------------------------------------------------------------------------------
namespace {

// the entry of global slot s (< the index length), copied from the device whose segment holds it
int read_entry(csvb200_multi_index* mi, uint64_t s, uint64_t* out)
{
    const uint32_t j = segment_of(mi->base.data(), (uint32_t)mi->seg.size(), s);
    csvb200_ctx* ctx = mi->m->ctx[j];
    CU_TRY(ctx, cudaSetDevice(ctx->device));
    CU_TRY(ctx, cudaMemcpyAsync(out, mi->table.ptr[j] + (s - mi->base[j]), sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return CSVB200_OK;
}

int first_device_error(csvb200_multi* m, const std::vector<int>& rcs)
{
    for (size_t k = 0; k < rcs.size(); ++k)
        if (rcs[k]) return mfail(m, rcs[k], "device " + std::to_string(k) + ": " + csvb200_last_error(m->ctx[k]));
    return CSVB200_OK;
}

}  // namespace

extern "C" {

int csvb200_multi_tape_validate(csvb200_multi_index* mi, uint32_t field_cnt, int crlf, csvb200_tape_report* out)
{
    if (!mi || !out) return CSVB200_ERR_INVALID_ARG;
    csvb200_multi* m = mi->m;
    const uint64_t len = mi->base.back();
    const uint64_t j = crlf ? (uint64_t)field_cnt + 1 : (uint64_t)field_cnt;   // src/tape.rs:318-321
    if (j == 0 || len == 0) return mfail(m, CSVB200_ERR_INVALID_ARG, "field_cnt must be >= 1");
    const int G = (int)mi->seg.size();
    // device k checks the global slots [max(1, base[k]), base[k + 1]) of its segment against its shard.  The LF slot of a
    // CRLF file compares its entry with the one before it, which for a segment's first slot lives in the nearest lower
    // non-empty segment (slot 0 for segment 0): read here, one entry per segment, and handed to the kernel.
    std::vector<uint64_t> prev(G, 0);
    for (int k = 0; k < G && crlf; ++k) {
        const uint64_t first = std::max<uint64_t>(1, mi->base[k]);
        if (first < mi->base[k + 1]) {
            int rc = read_entry(mi, first - 1, &prev[k]);
            if (rc) return mfail(m, rc, csvb200_last_error(m->ctx[segment_of(mi->base.data(), (uint32_t)G, first - 1)]));
        }
    }
    std::vector<int> rcs(G, CSVB200_OK);
    std::vector<uint64_t> bad(G, UINT64_MAX);
    run_phase(m, [&](int k) {
        csvb200_ctx* ctx = m->ctx[k];
        rcs[k] = [&]() -> int {
            const uint64_t first = std::max<uint64_t>(1, mi->base[k]);
            if (first >= mi->base[k + 1]) return CSVB200_OK;
            CU_TRY(ctx, cudaSetDevice(ctx->device));
            CellLease lease(ctx, 1);
            if (!lease.ok()) return fail(ctx, CSVB200_ERR_OOM, "no free result cell (4095 live index objects)");
            uint64_t* d_cell = ctx->d_cells + lease.first * kCellWords;
            uint64_t* h_cell = ctx->h_cells + lease.first * kCellWords;
            CU_TRY(ctx, cudaMemsetAsync(d_cell, 0xff, sizeof(uint64_t), ctx->stream));
            TapeValidateParams p{};
            p.index = by_global_slot(mi->table.ptr[k], mi->base[k]);
            p.entry_bytes = 8;
            p.index_len = mi->base[k + 1];
            p.bytes = mi->d_bytes[k];
            p.n = mi->cuts[k + 1] - mi->cuts[k];
            p.pos_bias = mi->cuts[k];
            p.jump = j;
            p.crlf = crlf ? 1 : 0;
            p.first_bad_slot = d_cell;
            p.first_slot = first;
            p.prev_entry = prev[k];
            CU_TRY(ctx, launch_tape_validate_segment(p, ctx->stream));
            ctx->launches += 1;
            CU_TRY(ctx, cudaMemcpyAsync(h_cell, d_cell, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            bad[k] = h_cell[0];
            return CSVB200_OK;
        }();
    });
    int rc = first_device_error(m, rcs);
    if (rc) return rc;
    std::memset(out, 0, sizeof(*out));
    out->index_len = len;
    out->jump = j;
    out->record_cnt = (uint32_t)((len - 1) / j);   // src/tape.rs:323-325
    out->problem = (len - 1) % j;                  // src/tape.rs:327
    out->first_bad_slot = *std::min_element(bad.begin(), bad.end());
    out->first_bad_record = UINT64_MAX;
    out->first_bad_pos = UINT64_MAX;
    if (out->first_bad_slot != UINT64_MAX) {
        out->first_bad_record = (out->first_bad_slot - 1) / j;
        rc = read_entry(mi, out->first_bad_slot, &out->first_bad_pos);
        if (rc) return mfail(m, rc, csvb200_last_error(m->ctx[segment_of(mi->base.data(), (uint32_t)G, out->first_bad_slot)]));
    } else if (out->problem != 0) {
        out->first_bad_record = (len - 1) / j;     // the file ends inside this record
    }
    out->ok = out->first_bad_slot == UINT64_MAX && out->problem == 0;
    return CSVB200_OK;
}

int csvb200_multi_validate_utf8(csvb200_multi_index* mi, uint64_t* valid_up_to, int* is_ascii)
{
    if (!mi) return CSVB200_ERR_INVALID_ARG;
    csvb200_multi* m = mi->m;
    const int G = (int)mi->seg.size();
    // the first and last (up to) 3 bytes of every shard, from which the host assembles every shard's halo
    std::vector<uint8_t> first3(3 * G, 0), last3(3 * G, 0);
    std::vector<int> rcs(G, CSVB200_OK);
    run_phase(m, [&](int k) {
        csvb200_ctx* ctx = m->ctx[k];
        rcs[k] = [&]() -> int {
            const size_t n = mi->cuts[k + 1] - mi->cuts[k], c = std::min<size_t>(3, n);
            if (c == 0) return CSVB200_OK;
            uint8_t tail[3];
            CU_TRY(ctx, cudaSetDevice(ctx->device));
            CU_TRY(ctx, cudaMemcpyAsync(&first3[3 * k], mi->d_bytes[k], c, cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaMemcpyAsync(tail, mi->d_bytes[k] + n - c, c, cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            for (size_t i = 0; i < c; ++i) last3[3 * k + i] = tail[c - 1 - i];
            return CSVB200_OK;
        }();
    });
    int rc = first_device_error(m, rcs);
    if (rc) return rc;
    std::vector<uint64_t> bad(G, UINT64_MAX), high(G, 0);
    run_phase(m, [&](int k) {
        csvb200_ctx* ctx = m->ctx[k];
        rcs[k] = [&]() -> int {
            const uint64_t n = mi->cuts[k + 1] - mi->cuts[k];
            if (n == 0) return CSVB200_OK;
            const Utf8Halo halo = utf8_halo(mi->cuts.data(), (uint32_t)G, (uint32_t)k,
                                            reinterpret_cast<const uint8_t(*)[3]>(first3.data()),
                                            reinterpret_cast<const uint8_t(*)[3]>(last3.data()));
            CU_TRY(ctx, cudaSetDevice(ctx->device));
            CellLease lease(ctx, 1);
            if (!lease.ok()) return fail(ctx, CSVB200_ERR_OOM, "no free result cell (4095 live index objects)");
            uint64_t* d_cell = ctx->d_cells + lease.first * kCellWords;
            uint64_t* h_cell = ctx->h_cells + lease.first * kCellWords;
            CU_TRY(ctx, cudaMemsetAsync(d_cell, 0xff, sizeof(uint64_t), ctx->stream));
            CU_TRY(ctx, cudaMemsetAsync(d_cell + 1, 0, sizeof(uint64_t), ctx->stream));
            CU_TRY(ctx, launch_utf8_validate_segment(mi->d_bytes[k], n, mi->cuts[k], halo, d_cell, ctx->stream));
            ctx->launches += 1;
            CU_TRY(ctx, cudaMemcpyAsync(h_cell, d_cell, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            bad[k] = h_cell[0];
            high[k] = h_cell[1];
            return CSVB200_OK;
        }();
    });
    rc = first_device_error(m, rcs);
    if (rc) return rc;
    if (valid_up_to) *valid_up_to = *std::min_element(bad.begin(), bad.end());
    if (is_ascii) *is_ascii = *std::max_element(high.begin(), high.end()) ? 0 : 1;
    return CSVB200_OK;
}

int csvb200_multi_tape_chunks(csvb200_multi_index* mi, uint8_t num, csvb200_chunk* out, size_t out_cap, size_t* n_out)
{
    if (!mi || !n_out) return CSVB200_ERR_INVALID_ARG;
    csvb200_multi* m = mi->m;
    if (!mi->tape_ready) return mfail(m, CSVB200_ERR_INVALID_STATE, "csvb200_multi_tape_init has not been called");
    int rc = tape_chunk_slots(mi->record_cnt, mi->jump, num, out, out_cap, n_out);
    if (rc) return mfail(m, rc, tape_chunk_error(rc));
    // the byte ranges: two entries per chunk, each gathered on the device whose segment holds it
    const int G = (int)mi->seg.size();
    const size_t nvals = 2 * *n_out;
    std::vector<uint64_t> slots(nvals), vals(nvals, UINT64_MAX);
    std::vector<uint32_t> owner(nvals);
    for (size_t i = 0; i < *n_out; ++i) {
        slots[2 * i] = out[i].start;
        slots[2 * i + 1] = out[i].end;
    }
    for (size_t i = 0; i < nvals; ++i) owner[i] = segment_of(mi->base.data(), (uint32_t)G, slots[i]);
    std::vector<int> rcs(G, CSVB200_OK);
    run_phase(m, [&](int k) {
        csvb200_ctx* ctx = m->ctx[k];
        rcs[k] = [&]() -> int {
            std::vector<uint64_t> local, got;
            for (size_t i = 0; i < nvals; ++i)
                if (owner[i] == (uint32_t)k) local.push_back(slots[i] - mi->base[k]);
            if (local.empty()) return CSVB200_OK;
            got.resize(local.size());
            CU_TRY(ctx, cudaSetDevice(ctx->device));
            DevBuf d_slots, d_vals;
            CU_TRY(ctx, d_slots.alloc(local.size() * 8, ctx->stream));
            CU_TRY(ctx, d_vals.alloc(local.size() * 8, ctx->stream));
            CU_TRY(ctx, cudaMemcpyAsync(d_slots.p, local.data(), local.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
            CU_TRY(ctx, launch_gather_slots(mi->table.ptr[k], 8, mi->base[k + 1] - mi->base[k], d_slots.as<uint64_t>(),
                                            local.size(), d_vals.as<uint64_t>(), ctx->stream));
            ctx->launches += 1;
            CU_TRY(ctx, cudaMemcpyAsync(got.data(), d_vals.p, got.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
            CU_TRY(ctx, cudaStreamSynchronize(ctx->stream));
            for (size_t i = 0, q = 0; i < nvals; ++i)
                if (owner[i] == (uint32_t)k) vals[i] = got[q++];
            return CSVB200_OK;
        }();
    });
    rc = first_device_error(m, rcs);
    if (rc) return rc;
    for (size_t i = 0; i < *n_out; ++i) {
        out[i].byte_start = vals[2 * i] == UINT64_MAX ? UINT64_MAX : vals[2 * i] + 1;
        out[i].byte_end = vals[2 * i + 1] == UINT64_MAX ? UINT64_MAX : vals[2 * i + 1] + 1;
    }
    return CSVB200_OK;
}

}  // extern "C"
