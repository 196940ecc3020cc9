// materialize.cu -- K6: column materialisation (SURVEY 8f rank 2).
//
// RecordSource::seek_field (src/record_source.rs:104-140) hands back the RAW slice of a field,
// "incl. surrounding quotes / padding; no unescape, no trim" (:135-139).  What callers do next is turn
// a column of such slices into values; this file does that on the device for a whole column at once:
//   for r in [first_record, first_record + nrec):   (start, end) = seek_field(r, field_idx)
//       value = raw slice, optionally trimmed of ASCII space / tab, optionally RFC-4180 unquoted
//               (outer quotes stripped when both are present, "" -> ")
//   offsets[r - first_record] = exclusive prefix sum of the value lengths, out = values back to back
// Two kernels: (1) lengths + exclusive scan fused (one pass, decoupled look-back over 62-bit sums),
// (2) the write.  Both read two index entries per record and the field's bytes: HBM sector-bound.
#include "internal.h"

namespace csvb200 {

namespace {

constexpr int kMatThreads = 256;
constexpr int kMatItems = 4;
constexpr int kMatTile = kMatThreads * kMatItems;
constexpr uint64_t kMatAgg = 1ull << 62, kMatPrefix = 2ull << 62, kMatMask = (1ull << 62) - 1;

__device__ __forceinline__ uint64_t ldg_u64(const uint64_t* p)
{
    uint64_t v;
    asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint64_t ld_relaxed(const uint64_t* p)
{
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed(uint64_t* p, uint64_t v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Decoupled look-back by one thread over the tile totals (status in the top two bits): publishes this tile's total,
// sums the totals of the tiles before it back to the nearest published prefix, publishes prefix + total and returns the
// prefix.  Tiles must be taken in ticket order.
__device__ __forceinline__ uint64_t lookback(uint64_t* desc, uint32_t tile, uint64_t total)
{
    st_relaxed(desc + tile, kMatAgg | (total & kMatMask));
    uint64_t prefix = 0;
    for (int64_t t = (int64_t)tile - 1; t >= 0;) {
        const uint64_t d = ld_relaxed(desc + t);
        const uint64_t st = d >> 62;
        if (st == 0) {
            __nanosleep(40);
            continue;
        }
        prefix += d & kMatMask;
        if (st == 2) break;
        --t;
    }
    st_relaxed(desc + tile, kMatPrefix | ((prefix + total) & kMatMask));
    return prefix;
}

// what the per-value helpers need of either parameter block
struct FieldView {
    const uint64_t* index;
    uint64_t index_len;
    const uint8_t* bytes;
    uint64_t n, pos_bias;
    uint32_t record_cnt, field_cnt, row_size, field_idx, flags;
};
__device__ __forceinline__ FieldView view_of(const MaterializeParams& p)
{
    return FieldView{p.index, p.index_len, p.bytes, p.n, p.pos_bias, p.record_cnt, p.field_cnt, p.row_size, p.field_idx, p.flags};
}
__device__ __forceinline__ FieldView view_of(const MaterializeMultiParams& p, uint32_t c)
{
    return FieldView{p.index, p.index_len, p.bytes, p.n, p.pos_bias, p.record_cnt, p.field_cnt, p.row_size, p.field_idx[c], p.flags};
}

// seek_field (src/record_source.rs:104-140) as byte offsets relative to p.bytes; false = Ok(None) or a
// slot the reference would panic on
__device__ __forceinline__ bool field_range(const FieldView& p, uint32_t r, uint64_t& a, uint64_t& b)
{
    if ((uint32_t)(r + 1u) >= p.record_cnt || p.field_idx >= p.field_cnt) return false;
    const uint32_t s = (uint32_t)(r + 1u) * p.row_size + p.field_idx;   // u32 arithmetic, as the reference
    if ((uint64_t)s + 1 >= p.index_len) return false;
    a = ldg_u64(p.index + s) + 1 - p.pos_bias;
    b = ldg_u64(p.index + s + 1) - p.pos_bias;
    return a <= b && b <= p.n;
}

// trims [a, b) in place and reports whether the value is a quoted field to unquote
__device__ __forceinline__ bool trim_and_test(const FieldView& p, uint64_t& a, uint64_t& b)
{
    const uint8_t* x = p.bytes;
    if (p.flags & 2u) {
        while (a < b && (x[a] == 0x20u || x[a] == 0x09u)) ++a;
        while (b > a && (x[b - 1] == 0x20u || x[b - 1] == 0x09u)) --b;
    }
    if ((p.flags & 1u) && b - a >= 2 && x[a] == 0x22u && x[b - 1] == 0x22u) {
        ++a;
        --b;
        return true;
    }
    return false;
}

__device__ __forceinline__ uint4 ldg_128(const void* p)
{
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// Calls f(byte) for every byte of x[a, b) in order, fetching the range as aligned 16-byte words: two or three
// 128-bit loads per value instead of one byte load per character (with 64 warps per SM each walking a different
// 128-byte line, byte-at-a-time loads thrash L1 and every character becomes an L2 round trip).  x must be 16-byte
// aligned (the ABI requires it of device inputs); a chunk that would read past n is fetched bytewise.
template <class F>
__device__ __forceinline__ void scan_bytes(const uint8_t* __restrict__ x, uint64_t n, uint64_t a, uint64_t b, F&& f)
{
    for (uint64_t base = a & ~15ull; base < b; base += 16) {
        uint32_t w[4];
        if (base + 16 <= n) {
            const uint4 v = ldg_128(x + base);
            w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint32_t t = 0;
                for (int j = 0; j < 4; ++j)
                    if (base + 4 * k + j < n) t |= (uint32_t)x[base + 4 * k + j] << (8 * j);
                w[k] = t;
            }
        }
        const uint32_t lo = a > base ? (uint32_t)(a - base) : 0u;
        const uint32_t hi = b - base < 16 ? (uint32_t)(b - base) : 16u;
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if ((uint32_t)k >= lo && (uint32_t)k < hi) f((w[k >> 2] >> (8 * (k & 3))) & 0xffu);
    }
}

// RFC-4180 unquoting as a streaming rule: a quote is held back one byte; a second quote right after it turns the
// pair into one '"', anything else releases the held quote as it is (same result as the scalar definition: '"'
// followed by '"' emits one and skips both, a lone '"' stays).
template <class Emit>
struct Unquoter {
    Emit emit;
    bool held = false;
    __device__ __forceinline__ void operator()(uint32_t c)
    {
        if (held) {
            held = false;
            emit(0x22u);
            if (c == 0x22u) return;
        }
        if (c == 0x22u)
            held = true;
        else
            emit(c);
    }
    __device__ __forceinline__ void finish()
    {
        if (held) emit(0x22u);
        held = false;
    }
};

// length of the value made of the raw slice [a, b)
__device__ __forceinline__ uint64_t value_len_range(const FieldView& p, uint64_t a, uint64_t b)
{
    if (!trim_and_test(p, a, b)) return b - a;
    uint64_t o = 0;
    auto count = [&](uint32_t) { ++o; };
    Unquoter<decltype(count)> u{count};
    scan_bytes(p.bytes, p.n, a, b, u);
    u.finish();
    return o;
}

__device__ __forceinline__ uint64_t value_len(const FieldView& p, uint32_t r)
{
    uint64_t a, b;
    if (!field_range(p, r, a, b)) return 0;
    return value_len_range(p, a, b);
}

// put(byte) for every byte of the value made of the raw slice [a, b); x is the caller's restrict-qualified copy of
// p.bytes (without it every byte load has to wait for the previous byte store)
template <class Put>
__device__ __forceinline__ void emit_value(const FieldView& p, const uint8_t* __restrict__ x, uint64_t a, uint64_t b, Put put)
{
    if (!trim_and_test(p, a, b)) {
        if (b - a < 16) {   // short raw values: a handful of byte loads beat 16 predicated steps per chunk
            for (; a < b; ++a) put(x[a]);
        } else {
            scan_bytes(x, p.n, a, b, put);
        }
    } else {
        Unquoter<Put> u{put};
        scan_bytes(x, p.n, a, b, u);
        u.finish();
    }
}

constexpr int kColBatch = 4;
constexpr uint32_t kColBatchMin = 8;   // columns from which the batched form pays

__device__ __forceinline__ uint32_t ldg_u8(const uint8_t* p)
{
    uint32_t v;
    asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// The dependent chain of one value is index slots -> first / last byte -> (only for padded or quoted values) a walk.
// A thread that resolves the columns of its row issues each level for a batch of kColBatch columns before it uses any of
// them: kColBatch loads in flight per thread instead of one round trip after another (1 GiB unquoted, 8 / 16 columns:
// 3.43 -> 3.00 ms, 6.83 -> 4.82 ms; batches of 8 cost 80 registers and lose it again; the single-column kernels are
// DRAM-sector-bound at 0.75-0.89 of peak and gain nothing from it).  ok bit k: the value exists;
// plain bit k: neither end is padding and it is not a quoted field, so the value IS the raw slice [a, b).
template <int kB>
struct RangeBatch {
    uint64_t a[kB], b[kB];
    uint32_t ok, plain, quoted;   // quoted bit k: not padded, both ends are quotes: the value is the unquoted [a + 1, b - 1)
};
// item(k, rec, fld) -> does item k exist, and which (record, field) it is
template <int kB, class Item>
__device__ __forceinline__ void range_batch_load(const FieldView& p, Item item, RangeBatch<kB>& rb)
{
    rb.ok = rb.plain = rb.quoted = 0;
#pragma unroll
    for (int k = 0; k < kB; ++k) {
        rb.a[k] = rb.b[k] = 0;
        uint32_t r = 0, f = 0;
        if (!item(k, r, f)) continue;
        if ((uint32_t)(r + 1u) >= p.record_cnt || f >= p.field_cnt) continue;
        const uint32_t s = (uint32_t)(r + 1u) * p.row_size + f;   // u32 arithmetic, as the reference
        if ((uint64_t)s + 1 >= p.index_len) continue;
        rb.a[k] = ldg_u64(p.index + s);
        rb.b[k] = ldg_u64(p.index + s + 1);
        rb.ok |= 1u << k;
    }
#pragma unroll
    for (int k = 0; k < kB; ++k) {
        if (!(rb.ok >> k & 1u)) continue;
        rb.a[k] = rb.a[k] + 1 - p.pos_bias;
        rb.b[k] = rb.b[k] - p.pos_bias;
        if (!(rb.a[k] <= rb.b[k] && rb.b[k] <= p.n)) rb.ok &= ~(1u << k);
    }
    if (p.flags == 0u) {
        rb.plain = rb.ok;
        return;
    }
    uint32_t fb[kB], lb[kB];
#pragma unroll
    for (int k = 0; k < kB; ++k) {
        fb[k] = lb[k] = 0;
        if ((rb.ok >> k & 1u) && rb.b[k] > rb.a[k]) {
            fb[k] = ldg_u8(p.bytes + rb.a[k]);
            lb[k] = ldg_u8(p.bytes + rb.b[k] - 1);
        }
    }
#pragma unroll
    for (int k = 0; k < kB; ++k) {
        if (!(rb.ok >> k & 1u)) continue;
        const bool padded = (p.flags & 2u) && (fb[k] == 0x20u || fb[k] == 0x09u || lb[k] == 0x20u || lb[k] == 0x09u);
        const bool quoted = (p.flags & 1u) && rb.b[k] - rb.a[k] >= 2 && fb[k] == 0x22u && lb[k] == 0x22u;
        if (rb.b[k] == rb.a[k] || (!padded && !quoted)) rb.plain |= 1u << k;
        else if (!padded) rb.quoted |= 1u << k;
    }
}

__global__ void __launch_bounds__(kMatThreads) materialize_offsets_kernel(const MaterializeParams p)
{
    __shared__ uint64_t s_warp[kMatThreads / 32];
    __shared__ uint64_t s_prefix;
    __shared__ uint32_t s_tile;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(p.ticket, 1u);   // tiles are taken in order: look-back only waits on started tiles
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t i0 = (uint64_t)tile * kMatTile + (uint64_t)tid * kMatItems;
    uint64_t len[kMatItems], tsum = 0;
#pragma unroll
    for (int k = 0; k < kMatItems; ++k) {
        len[k] = i0 + k < p.nrec ? value_len(view_of(p), p.first_record + (uint32_t)(i0 + k)) : 0;
        tsum += len[k];
    }
    // block exclusive scan of the thread sums
    uint64_t inc = tsum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint64_t v = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (uint32_t)d) inc += v;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    uint64_t wbase = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kMatThreads / 32; ++w) {
        if (w < (int)warp) wbase += s_warp[w];
        total += s_warp[w];
    }
    if (tid == 0) s_prefix = lookback(p.tile_desc, tile, total);
    __syncthreads();
    uint64_t off = p.offset_base + s_prefix + wbase + (inc - tsum);
#pragma unroll
    for (int k = 0; k < kMatItems; ++k) {
        if (i0 + k < p.nrec) p.offsets[i0 + k] = off;
        off += len[k];
    }
    if (i0 < p.nrec && i0 + kMatItems >= p.nrec) p.offsets[p.nrec] = off;   // the thread owning the last record
}

__global__ void __launch_bounds__(kMatThreads) materialize_write_kernel(const MaterializeParams p)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    // restrict-qualified local copies: without them every byte load has to wait for the previous byte store
    // (the compiler must assume out aliases bytes), which serialises the copy into load -> store round trips
    const uint8_t* __restrict__ x = p.bytes;
    uint8_t* __restrict__ out = p.out;
    const FieldView fv = view_of(p);
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p.nrec; i += stride) {
        uint64_t a, b;
        if (!field_range(fv, p.first_record + (uint32_t)i, a, b)) continue;
        uint64_t o = p.offsets[i];
        const uint64_t o_end = p.offsets[i + 1];
        if (o_end > p.out_cap) continue;   // host form checks the capacity first; device form clips whole values
        emit_value(fv, x, a, b, [&](uint32_t c) { out[o++] = (uint8_t)c; });
    }
}

// ---- several columns in one sweep --------------------------------------------------------------------------------
// A tile is 256 consecutive records, one per thread; the thread walks the requested fields of ITS row, so the index
// slots and bytes of neighbouring columns come out of the sectors the first column fetched.  Per column: a block scan
// of the 256 lengths (warp w scans columns w, w + 8, ...), one decoupled look-back chain over the tile totals
// (thread c looks back for column c), then the exclusive offsets go out coalesced.
// A row sweep (tiles of 32-128 records staged through shared memory) was built, measured against these kernels and
// removed: it won on quoted columns and lost on unquoted ones (DESIGN 4.8, profiles/r02_mat_sweep_ab.jsonl).
using ColBatch = RangeBatch<kColBatch>;
__device__ __forceinline__ void col_batch_load(const MaterializeMultiParams& p, uint32_t r, uint32_t c0, bool row_live, ColBatch& cb)
{
    range_batch_load(view_of(p, 0), [&](int k, uint32_t& rec, uint32_t& fld) {
        const uint32_t c = c0 + (uint32_t)k;
        if (!row_live || c >= p.ncols) return false;
        rec = r;
        fld = p.field_idx[c];
        return true;
    }, cb);
}

template <bool kBatched>   // separate kernels: the batched form needs 64 registers, the plain one 32
__global__ void __launch_bounds__(kMultiThreads) materialize_multi_offsets_kernel(const MaterializeMultiParams p)
{
    extern __shared__ uint32_t s_len[];                    // [ncols][256] lengths, then exclusive prefixes in place
    __shared__ uint64_t s_total[kMatMaxCols], s_base[kMatMaxCols];
    __shared__ uint32_t s_tile;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(p.ticket, 1u);        // tiles are taken in order: look-back only waits on started tiles
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t i = (uint64_t)tile * kMultiThreads + tid;
    // fewer than kColBatchMin columns: one value after the other (the batches cost registers: 4 columns 1.86 -> 2.01 ms
    // unquoted, 3.01 -> 3.29 ms quoted, where 8 / 16 unquoted columns go 3.43 -> 2.96 ms and 6.83 -> 4.74 ms)
    for (uint32_t c = 0; !kBatched && c < p.ncols; ++c)
        s_len[c * kMultiThreads + tid] = i < p.nrec ? (uint32_t)value_len(view_of(p, c), p.first_record + (uint32_t)i) : 0u;
    for (uint32_t c0 = 0; kBatched && c0 < p.ncols; c0 += kColBatch) {
        ColBatch cb;
        col_batch_load(p, p.first_record + (uint32_t)i, c0, i < p.nrec, cb);
#pragma unroll
        for (int k = 0; k < kColBatch; ++k) {
            const uint32_t c = c0 + (uint32_t)k;
            if (c >= p.ncols) break;
            uint32_t len = 0;
            if (cb.plain >> k & 1u)
                len = (uint32_t)(cb.b[k] - cb.a[k]);
            else if (cb.quoted >> k & 1u) {
                uint32_t o = 0;
                auto count = [&](uint32_t) { ++o; };
                Unquoter<decltype(count)> u{count};
                scan_bytes(p.bytes, p.n, cb.a[k] + 1, cb.b[k] - 1, u);
                u.finish();
                len = o;
            } else if (cb.ok >> k & 1u)
                len = (uint32_t)value_len_range(view_of(p, c), cb.a[k], cb.b[k]);          // padded: trim first
            s_len[c * kMultiThreads + tid] = len;
        }
    }
    __syncthreads();
    for (uint32_t c = warp; c < p.ncols; c += kMultiThreads / 32) {
        uint32_t* col = s_len + c * kMultiThreads;
        uint32_t v[8], sum = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            v[k] = col[8 * lane + k];
            sum += v[k];
        }
        uint32_t inc = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= (uint32_t)d) inc += t;
        }
        uint32_t run = inc - sum;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            col[8 * lane + k] = run;
            run += v[k];
        }
        if (lane == 31) s_total[c] = inc;
    }
    __syncthreads();
    // one chain per column, thread c walks column c's: all the chains of the tile advance together in one warp
    // (a warp per chain with 128-descriptor hops measured slower here: 0.404 against 0.362 ms for 8 columns, 0.697
    // against 0.513 ms for 16 -- with 256-row tiles the walks are short and the chains queue up)
    if (tid < p.ncols) s_base[tid] = p.offset_base[tid] + lookback(p.tile_desc + (uint64_t)tid * p.tiles, tile, s_total[tid]);
    __syncthreads();
    for (uint32_t c = 0; c < p.ncols; ++c) {
        const uint64_t off = s_base[c] + s_len[c * kMultiThreads + tid];
        if (i < p.nrec) p.offsets[c][i] = off;
        if (i + 1 == p.nrec) p.offsets[c][p.nrec] = s_base[c] + s_total[c];   // the thread owning the last record
    }
}

template <bool kBatched>
__global__ void __launch_bounds__(kMultiThreads) materialize_multi_write_kernel(const MaterializeMultiParams p)
{
    const uint8_t* __restrict__ x = p.bytes;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.nrec) return;
    for (uint32_t c = 0; !kBatched && c < p.ncols; ++c) {
        const FieldView fv = view_of(p, c);
        uint8_t* __restrict__ out = p.out[c];
        uint64_t a, b;
        if (!field_range(fv, p.first_record + (uint32_t)i, a, b)) continue;
        uint64_t o = p.offsets[c][i];
        if (p.offsets[c][i + 1] > p.out_cap[c]) continue;
        emit_value(fv, x, a, b, [&](uint32_t ch) { out[o++] = (uint8_t)ch; });
    }
    for (uint32_t c0 = 0; kBatched && c0 < p.ncols; c0 += kColBatch) {
        ColBatch cb;
        col_batch_load(p, p.first_record + (uint32_t)i, c0, true, cb);
        uint64_t o[kColBatch], o_end[kColBatch];
#pragma unroll
        for (int k = 0; k < kColBatch; ++k) {
            o[k] = o_end[k] = 0;
            if (cb.ok >> k & 1u) {
                o[k] = p.offsets[c0 + k][i];
                o_end[k] = p.offsets[c0 + k][i + 1];
            }
        }
#pragma unroll
        for (int k = 0; k < kColBatch; ++k) {
            const uint32_t c = c0 + (uint32_t)k;
            if (c >= p.ncols) break;
            if (!(cb.ok >> k & 1u) || o_end[k] > p.out_cap[c]) continue;   // the device form clips whole values
            uint8_t* __restrict__ out = p.out[c];
            uint64_t at = o[k];
            auto put = [&](uint32_t ch) { out[at++] = (uint8_t)ch; };
            uint64_t a = cb.a[k], b = cb.b[k];
            if (cb.plain >> k & 1u) {
                if (b - a < 16) {   // short raw values: a handful of byte loads beat 16 predicated steps per chunk
                    for (; a < b; ++a) put(x[a]);
                } else {
                    scan_bytes(x, p.n, a, b, put);
                }
                continue;
            }
            if (cb.quoted >> k & 1u) {
                Unquoter<decltype(put)> u{put};
                scan_bytes(x, p.n, a + 1, b - 1, u);
                u.finish();
                continue;
            }
            emit_value(view_of(p, c), x, a, b, put);   // padded: trim first
        }
    }
}

}  // namespace

size_t materialize_multi_scratch_bytes(uint32_t nrec, uint32_t ncols)
{
    const size_t tiles = ((size_t)nrec + kMultiThreads - 1) / kMultiThreads + 1;
    return 128 + tiles * ncols * sizeof(uint64_t);
}

cudaError_t launch_materialize_multi_offsets(const MaterializeMultiParams& p, cudaStream_t stream)
{
    if (p.tiles == 0 || p.ncols == 0) return cudaSuccess;
    const size_t smem = (size_t)p.ncols * kMultiThreads * sizeof(uint32_t);
    if (p.ncols >= kColBatchMin)
        materialize_multi_offsets_kernel<true><<<p.tiles, kMultiThreads, smem, stream>>>(p);
    else
        materialize_multi_offsets_kernel<false><<<p.tiles, kMultiThreads, smem, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_materialize_multi_write(const MaterializeMultiParams& p, cudaStream_t stream)
{
    if (p.nrec == 0 || p.ncols == 0) return cudaSuccess;
    const unsigned blocks = (p.nrec + kMultiThreads - 1) / kMultiThreads;
    if (p.ncols >= kColBatchMin)
        materialize_multi_write_kernel<true><<<blocks, kMultiThreads, 0, stream>>>(p);
    else
        materialize_multi_write_kernel<false><<<blocks, kMultiThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

size_t materialize_scratch_bytes(uint32_t nrec) { return 128 + ((size_t)(nrec + kMatTile - 1) / kMatTile + 1) * sizeof(uint64_t); }

cudaError_t launch_materialize_offsets(const MaterializeParams& p, cudaStream_t stream)
{
    const uint32_t tiles = (p.nrec + kMatTile - 1) / kMatTile;
    if (tiles == 0) return cudaSuccess;
    materialize_offsets_kernel<<<tiles, kMatThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_materialize_write(const MaterializeParams& p, cudaStream_t stream)
{
    if (p.nrec == 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint64_t blocks = ((uint64_t)p.nrec + kMatThreads - 1) / kMatThreads;
    const uint64_t max_blocks = (uint64_t)sms * 16;
    if (blocks > max_blocks) blocks = max_blocks;
    materialize_write_kernel<<<(unsigned)blocks, kMatThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace csvb200
