// index_common.cuh -- device helpers shared by the two index-build kernels
// (index_build.cu: simple one-tile-per-CTA kernel; index_build_tma.cu: persistent TMA pipeline).
#pragma once
#include "bitslice.cuh"
#include "internal.h"

namespace csvb200 {

__device__ __forceinline__ uint64_t ld_relaxed_u64(const uint64_t* p)
{
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(uint64_t* p, uint64_t v)
{
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint4 ldg_stream_128(const void* p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_128(void* p, uint64_t a, uint64_t b)
{
    // .cs: the index is written once and never read by this kernel (0.3979 vs 0.4006 ms on cfg2 against the plain store)
    asm volatile("st.global.cs.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(a), "l"(b) : "memory");
}

__device__ __forceinline__ void st_relaxed_sys_u64(uint64_t* p, uint64_t v)
{
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint64_t ld_acquire_sys_u64(const uint64_t* p)
{
    uint64_t v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t ld_volatile_u64(const uint64_t* p)
{
    uint64_t v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t global_timer_ns()
{
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// One thread.  Posts this shard's row {entries under the carry it used, end parity, carry used, total separators}
// to (slot = epoch % kExRing, row = rank) of EVERY rank's mailbox over peer-mapped pointers, then waits on its OWN
// mailbox for the rows of the lower ranks and derives from them (exactly what verify_carry_kernel derives from an
// all-gathered array): the true carry-in parity of this shard (XOR of the lower shards' parities, parity = end ^ used),
// the entries the lower shards emit under THEIR true carries (flipping a carry swaps inside / outside separators, so
// the other count is total - entries), and whether this shard's guess was wrong.
static __device__ __noinline__ void exchange_post_and_resolve(const ExchangeArgs ex, uint64_t entries, uint64_t end_parity,
                                                       uint64_t used, uint64_t total)
{
    const uint64_t off = ((ex.epoch % kExRing) * kExMaxWorld) * kExRowWords;
    for (uint32_t r = 0; r < ex.world; ++r) {
        uint64_t* row = ex.peers[r] + off + (uint64_t)ex.rank * kExRowWords;
        row[0] = entries;
        row[1] = end_parity;
        row[2] = used;
        row[3] = total;
    }
    // ONE system-scope fence orders the payload stores above before all the epoch words below (a release store per peer
    // is a fence per peer: ~10 us at 8 ranks, measured as the step overhead of rank 0, which waits for nobody)
    __threadfence_system();
    for (uint32_t r = 0; r < ex.world; ++r)
        st_relaxed_sys_u64(ex.peers[r] + off + (uint64_t)ex.rank * kExRowWords + 4, ex.epoch);
    const uint64_t* mine = ex.peers[ex.rank] + off;
    const uint64_t t0 = global_timer_ns();
    uint64_t carry = 0ull, below = 0ull, err = 0ull;
    for (uint32_t j = 0; j < ex.rank && !err; ++j) {
        const uint64_t* row = mine + (uint64_t)j * kExRowWords;
        uint64_t e;
        while ((e = ld_acquire_sys_u64(row + 4)) != ex.epoch) {
            // a LARGER epoch: the writer lapped the ring (more than kExRing builds ahead of this rank)
            if (e > ex.epoch || global_timer_ns() - t0 > ex.timeout_ns) {
                err = 1ull;
                break;
            }
            __nanosleep(100);
        }
        if (err) break;
        const uint64_t cnt = ld_volatile_u64(row + 0), tot = ld_volatile_u64(row + 3);
        const uint64_t us = ld_volatile_u64(row + 2) & 1ull, en = ld_volatile_u64(row + 1) & 1ull;
        below += carry == us ? cnt : tot - cnt;
        carry ^= en ^ us;
    }
    const uint64_t redo = (!err && carry != (used & 1ull)) ? 1ull : 0ull;
    ex.out[0] = 0ull;
    ex.out[1] = carry;
    ex.out[2] = below | (err << 63);
    ex.out[3] = redo;
    if (ex.out_host != nullptr) {
        ex.out_host[0] = 0ull;
        ex.out_host[1] = carry;
        ex.out_host[2] = below | (err << 63);
        ex.out_host[3] = redo;
    }
}

struct WarpState {
    uint32_t par;   // quote parity of the warps before this one (relative to tile start)
    uint32_t off0;  // entries emitted by those warps if the tile is entered outside quotes
    uint32_t off1;  // ... if entered inside quotes
};

constexpr int kGroups = kBytesPerThread / 32;   // 32-byte bit-slice groups per thread
constexpr int kChunks = kBytesPerThread / 16;   // 16-byte chunks per thread

// Virtual predecessor of tile 0: the carry entering this launch, encoded as a prefix descriptor.
__device__ __forceinline__ uint64_t virtual_prefix_desc(const BuildParams& p)
{
    uint64_t carry_count = p.carry_count;
    uint32_t carry_parity = p.carry_parity;
    if (p.pdl_wait) asm volatile("griddepcontrol.wait;" ::: "memory");   // the predictor's cell is complete and visible
    if (p.carry != nullptr) {
        if (!p.carry_parity_only) carry_count = p.carry[0];
        carry_parity = (uint32_t)p.carry[1] & 1u;
    }
    if (p.shard_par != nullptr) {
        carry_parity = 0u;
        for (uint32_t j = 0; j < p.shard_rank; ++j) carry_parity ^= p.shard_par[j] & 1u;
    }
    return kStatusPrefix | ((uint64_t)p.desc_tag << kTagShift) | (carry_parity ? kParityBit : 0ull) | (carry_count & kCountMask);
}

// Called by the thread that resolved the LAST tile of a launch: entries emitted through the end of the
// launch, the quote parity after its last byte and (4-word form) the carry parity the launch used.
__device__ __forceinline__ void write_result(const BuildParams& p, uint64_t cend, uint32_t pend)
{
    p.result[0] = cend;
    p.result[1] = pend;
    if (p.result_host != nullptr) {
        p.result_host[0] = cend;
        p.result_host[1] = pend;
    }
    if (p.result2 != nullptr) {
        p.result2[0] = cend;
        p.result2[1] = pend;
        if (p.result2_words >= 3u) p.result2[2] = (virtual_prefix_desc(p) >> 61) & 1ull;
    }
}

// Called by one thread of every CTA when its look-back role is over (its separator total already added to
// *p.total_out): the LAST such CTA of the launch holds the complete {entries, end parity} and total and runs the exchange
// while other CTAs may still be compacting -- the NVLink round trip hides behind the tail of the launch.
__device__ __forceinline__ void exchange_if_last(const BuildParams& p)
{
    if (p.ex_done == nullptr) return;
    __threadfence();
    if (atomicAdd(p.ex_done, 1u) != gridDim.x - 1u) return;
    __threadfence();
    if (p.validate) {
        // every CTA has added its newline count / non-ASCII flag: publish them next to {entries, end parity}
        const uint64_t nl = ld_volatile_u64(reinterpret_cast<const uint64_t*>(p.nl_out));
        const uint64_t hi = *reinterpret_cast<volatile const uint32_t*>(p.hi_out);
        p.result[2] = hi;
        p.result[3] = nl;
        if (p.result_host != nullptr) {
            p.result_host[2] = hi;
            p.result_host[3] = nl;
        }
    }
    const uint64_t total = p.total_out != nullptr ? ld_volatile_u64(reinterpret_cast<const uint64_t*>(p.total_out)) : 0ull;
    // this CTA is the last user of the counters in the scratch head: zero for the next launch (there is no memset)
    *p.ex_done = 0u;
    if (p.scratch_totals) {
        if (p.total_out != nullptr) *p.total_out = 0ull;
        if (p.nl_out != nullptr) *p.nl_out = 0ull;
        if (p.hi_out != nullptr) *p.hi_out = 0u;
    }
    if (p.ex.peers == nullptr) return;
    const uint64_t entries = ld_volatile_u64(p.result + 0), endp = ld_volatile_u64(p.result + 1);
    const uint64_t used = (virtual_prefix_desc(p) >> 61) & 1ull;
    exchange_post_and_resolve(p.ex, entries, endp, used, total);
}

// Warp-parallel decoupled look-back over the monoid (p, c0, c1) (see index_build.cu header).
// Called by one full warp after the tile's own aggregate has been published; returns the quote
// parity entering the tile (pin) and the number of index entries emitted before it (base).
//
// kLookbackPerLane descriptors are inspected per lane and round trip, i.e. a window of
// 32 * kLookbackPerLane predecessor tiles.  All resident CTAs advance in near lock-step, so the
// nearest published prefix is typically one "wave" (= number of resident CTAs) of tiles back; a
// window that covers the whole wave resolves the look-back in about one L2 round trip instead of
// wave / 32 serial ones (ncu: >50 % of worker stalls were waits on this chain with a 64-tile window).
// Measured with tools/timeline.py (round 2, 1 GiB quote-heavy, 444 CTAs, a ticket every ~16 ns): a look-back takes 6.5-7.2 us
// -- about the slack one super-tile of skew gives it (7.3 us), so 40-50 % of the tiles make their workers wait, 0.75-1 us
// on average = 8-11 % of the kernel.  It is 6.5 round trips of 1.1 us each (L2 latency under the streaming load), of which
// 3.9 are retries: the aggregates of the tiles just before ours arrive on average 2.7 us AFTER our own (max of the 64
// before us; ticket -> aggregates takes 5.9 us +- 1.3).  Tried on that evidence, all slower or equal: a two-level walk
// (a tile with no prefix in its window publishes the composite of [tile - 32, tile]; later round trips read 32 such
// spans = 1056 tiles at once: 2 forward trips instead of 2.6 but more retries, 0.342 against 0.330 ms); every lane
// waiting for its own descriptor (no retries, 2.7 trips of 2.8 us: 0.337); 64 / 128 descriptors per trip with and
// without the single-descriptor re-poll (0.338 / 0.373); a look-back warp that has resolved its tile also publishing the
// prefixes of the next tiles whose aggregates are in (idempotent forward push: 0.333 against 0.331, kv22).  What is left
// is inherent to one pass: prefix(t) needs the slowest of the ~100 tiles in flight before t.
template <int kLookbackPerLane, bool kDbg = false>
__device__ __forceinline__ void decoupled_lookback(const BuildParams& p, uint32_t tile, uint32_t lane, uint32_t& pin_out,
                                                   uint64_t& base_out)
{
    uint32_t dbg_trips = 0, dbg_polls = 0;   // (kDbg) round trips in all, of which retries of a window
    auto virtual_prefix = [&]() -> uint64_t { return virtual_prefix_desc(p); };

    // Suffix composite S = (sp, sc0, sc1) of the tiles already absorbed (those nearest to us).
    // One round inspects a window of 32 * kLookbackPerLane predecessors: lane L owns the
    // kLookbackPerLane CONSECUTIVE tiles idx0 - L*kLookbackPerLane - j (j = 0 nearest) and folds
    // them with plain register arithmetic (no warp collectives); one set of ballots / reductions
    // then combines the 32 lane composites.  All loads of a round are in flight together.
    uint32_t sp = 0u;
    uint64_t sc0 = 0ull, sc1 = 0ull;
    int64_t idx0 = (int64_t)tile - 1;
    uint32_t pin = 0u;
    uint64_t base = 0ull;
    while (true) {
        if (kDbg) ++dbg_trips;
        uint64_t d[kLookbackPerLane];
#pragma unroll
        for (int j = 0; j < kLookbackPerLane; ++j) {
            const int64_t idx = idx0 - (int64_t)lane * kLookbackPerLane - j;
            d[j] = idx >= 0 ? ld_relaxed_u64(p.desc + idx * kDescStride) : virtual_prefix();
            if (((d[j] >> kTagShift) & kTagMask) != (uint64_t)p.desc_tag) d[j] = 0ull;   // another launch's word: not ready
        }
        // lane-local fold, nearest tile first: L <- agg(t_j) o L
        uint32_t lp_ = 0u, l0 = 0u, l1 = 0u;   // lane composite (parity, c0, c1)
        uint32_t stop = 0u;                    // 0 = all aggregates, 1 = met an unpublished tile, 2 = met a prefix
        uint64_t pd = 0ull;                    // the prefix descriptor, if met
#pragma unroll
        for (int j = 0; j < kLookbackPerLane; ++j) {
            const uint32_t status = (uint32_t)(d[j] >> 62);
            if (stop == 0u) {
                if (status == 1u) {
                    const uint32_t ap = (uint32_t)((d[j] >> 61) & 1ull);
                    const uint32_t a0 = (uint32_t)(d[j] & 0xfffffull), a1 = (uint32_t)((d[j] >> 20) & 0xfffffull);
                    const uint32_t n0 = a0 + (ap ? l1 : l0);
                    const uint32_t n1 = a1 + (ap ? l0 : l1);
                    l0 = n0;
                    l1 = n1;
                    lp_ ^= ap;
                } else {
                    stop = status == 2u ? 2u : 1u;
                    pd = d[j];
                }
            }
        }
        const uint32_t stopped = __ballot_sync(0xffffffffu, stop != 0u);
        const uint32_t ls = stopped ? (uint32_t)(__ffs(stopped) - 1) : 32u;   // nearest lane that stopped
        const uint32_t ls_stop = __shfl_sync(0xffffffffu, stop, (int)(ls & 31u));
        if (ls < 32u && ls_stop == 1u) {   // an unpublished tile lies before the nearest prefix: poll again
            if (kDbg) ++dbg_polls;
            // wait on THAT descriptor alone (one line instead of the whole window per poll: hundreds of look-back warps
            // poll at the same time and their traffic competes with the data streams in L2), then rescan; re-polling
            // the whole window measured 0.3-1.1 % slower on both 1 GiB inputs (kv18 / kv20)
            const int64_t widx = idx0 - (int64_t)ls * kLookbackPerLane - (kLookbackPerLane - 1);
            if (lane == 0 && widx >= 0) {
                while ((ld_relaxed_u64(p.desc + widx * kDescStride) >> 62) == 0ull) __nanosleep(32);
            }
            __syncwarp();
            continue;
        }
        // lanes 0..ls contribute (lane ls only the tiles nearer than its prefix)
        const bool in_win = lane <= ls;
        const uint32_t pj = in_win ? lp_ : 0u;
        const uint32_t bp = __ballot_sync(0xffffffffu, pj != 0u);
        // parity accumulated by the window tiles EARLIER than this lane's (= higher lanes)
        const uint32_t rel = __popc(bp & (0xfffffffeu << lane)) & 1u;
        const uint32_t w0j = in_win ? (rel ? l1 : l0) : 0u;
        const uint32_t w1j = in_win ? (rel ? l0 : l1) : 0u;
        const uint32_t W0 = __reduce_add_sync(0xffffffffu, w0j);
        const uint32_t W1 = __reduce_add_sync(0xffffffffu, w1j);
        const uint32_t Wp = __popc(bp) & 1u;
        // S <- W o S   (the window is earlier in the file than everything absorbed so far)
        const uint64_t n0 = (uint64_t)W0 + (Wp ? sc1 : sc0);
        const uint64_t n1 = (uint64_t)W1 + (Wp ? sc0 : sc1);
        sc0 = n0;
        sc1 = n1;
        sp ^= Wp;
        if (ls < 32u) {
            const uint64_t pref = __shfl_sync(0xffffffffu, pd, (int)ls);
            const uint32_t P = (uint32_t)((pref >> 61) & 1ull);
            pin = P ^ sp;
            base = (pref & kCountMask) + (P ? sc1 : sc0);
            break;
        }
        idx0 -= 32 * kLookbackPerLane;
    }
    pin_out = pin;
    base_out = base;
    if (kDbg && lane == 0) p.dbg[(uint64_t)tile * 8 + 6] |= ((uint64_t)dbg_trips << 48) | ((uint64_t)dbg_polls << 56);   // clock64 of the ticket keeps 48 bits
}

}  // namespace csvb200
