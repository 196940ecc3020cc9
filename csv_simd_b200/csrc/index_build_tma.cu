// index_build_tma.cu -- persistent, warp-specialised, TMA-fed version of the fused index build.
//
// Same algorithm and output as index_build.cu (see its header for the reference mapping:
// reader::read src/reader.rs:150-306, SimdInput::structure src/avx/stage1.rs:193-407,
// Stage1::crush_set_bits src/stage1.rs:162-296), re-organised around what bounds it on B200
// (every step below is backed by an ncu capture, see profiles/ and DESIGN.md):
//
//   * the CTA is persistent (2 per SM) and split into roles:
//       warps 0-7  workers : classify / scan / compact      (256 threads x 128 B = one 32 KiB sub-tile)
//       warp  8    producer: takes tickets, issues one TMA 2-D load per sub-tile
//                            (cp.async.bulk.tensor, SWIZZLE_128B, mbarrier complete_tx)
//       warp  9    look-back: scans the warp aggregates, publishes the descriptor, runs the
//                            warp-parallel decoupled look-back, hands (parity, base) to the workers
//   * a look-back descriptor covers a SUPER-TILE of kSub consecutive sub-tiles (64 KiB): the chain of
//     prefixes advances one 32-descriptor window per L2 round trip, so bytes per descriptor set the
//     chain's byte rate; with one descriptor per 32 KiB the kernel was chain-bound at ~2.4 TB/s;
//   * the compaction of super-tile k is skewed behind the classification of super-tile k+1, so the
//     look-back latency is covered by useful work instead of a barrier stall;
//   * every descriptor sits in its own 128-byte line (internal.h kDescStride): hundreds of CTAs poll
//     the same few hundred descriptors and packed descriptors serialise on a handful of L2 slices;
//   * the thread that resolves tile 0 writes the sentinel index[0] = 0 (src/reader.rs:216) and the one that resolves
//     the last tile writes {entries, end parity} both to the device cell and to its pinned host mirror, so a build is
//     ONE launch with no memset / copy nodes around it except the zeroing of the look-back scratch;
//   * the input is a 2-D tensor map [rows = n/128][128 B]; rows past the end are zero-filled by the
//     TMA unit, which reproduces the reference's zero padding of the last block
//     (src/avx/stage1.rs:54-88) for free; the sub-row tail (< 128 B) is patched in by one thread.
#include <cuda.h>

#include <mutex>

#include "index_common.cuh"

namespace csvb200 {

namespace {

constexpr int kBoxRows = 128;                    // rows of 128 B per TMA box (16 KiB)
constexpr uint32_t kInvalidTile = 0xffffffffu;

// Shape of one build of the kernel.  What differs between the shapes is how many CTAs fit on an SM
// (the kernel is issue-bound on quote-heavy input, so resident warps matter) and how the shared memory that
// buys them is found:
//   kMinBlocks  CTAs per SM the register allocation is held to (__launch_bounds__)
//   kStageBufs  staging buffers of the compaction: 2 = double buffered (one barrier per sub-tile),
//               1 = a second barrier per sub-tile before the buffer is written again
//   kStageCap   entries per staging buffer; denser sub-tiles take extra rounds
//   kSub        sub-tiles (32 KiB TMA boxes) per look-back descriptor: the chain of prefixes advances a window
//               of descriptors per L2 round trip, so bytes per descriptor set the chain's byte rate
//   kSkew       super-tiles classified ahead of the one being compacted (what hides the look-back latency)
//   kWorkers    worker warps per CTA (a sub-tile is kWorkers x 4 KiB; 16-bit staging offsets allow up to 16):
//               the cost of the look-back chain grows with the number of CTAs in flight, so the same number
//               of resident worker warps in fewer, larger CTAs shortens it
template <int kMinBlocks_, int kStageBufs_, int kStageCap_, int kSub_, int kSkew_ = 1, int kWorkers_ = 8, int kExpand_ = 0, int kLook_ = 1>
struct TmaShape {
    // look-back: descriptors per lane and round trip (window = 32 * kLook; 64 / 128 measured slower in both rounds, also
    // with the single-descriptor re-poll: kv18)
    static constexpr int kLook = kLook_;
    // expansion loop: 0 = two entries per trip + a tail for the odd one; (1 = one loop whose second store is predicated,
    // no tail, no trip count: measured, not kept;) 2 = that loop on sub-tiles with fewer than 3 entries per 32-byte group, else 0.  Measured (kv14 /
    // kv15, 1 GiB): cfg2 0.3776 / 0.3791 / 0.3736 ms, cfg3 0.3416 / 0.3337 / 0.3318 ms for 0 / 1 / 2.  Walking the bits
    // from the top (clz is one FLO where ffs is BREV + FLO) and filling the slots backwards: no change (kv16); the first
    // two entries of a group without a loop, the rest in one: 0.3496 against 0.3299 ms on cfg3 (kv17).
    static constexpr int kExpand = kExpand_;
    static constexpr int kWorkers = kWorkers_;
    static constexpr int kWorkerThreads = kWorkers_ * 32;
    static constexpr int kThreadsAll = kWorkerThreads + 64;    // + TMA producer warp + look-back warp
    static constexpr int kProducerWarp = kWorkers_;
    static constexpr int kLookbackWarp = kWorkers_ + 1;
    static constexpr int kTile = kWorkerThreads * kBytesPerThread;   // bytes per sub-tile
    static constexpr int kRows = kWorkerThreads;                      // 128-byte rows per sub-tile
    static constexpr int kBoxes = kRows / kBoxRows;                   // TMA loads per sub-tile
    static_assert(kWorkers_ % 4 == 0 && kWorkers_ <= 16, "sub-tiles are whole 16 KiB boxes and at most 64 KiB");
    static constexpr int kSkew = kSkew_;
    static constexpr int kRing = kSkew_ + 1;               // ring depth of the worker <-> look-back hand-off buffers
    static constexpr int kMinBlocks = kMinBlocks_;
    static constexpr int kStageBufs = kStageBufs_;
    static constexpr int kStageCap = kStageCap_;
    static constexpr int kSub = kSub_;
    static constexpr int kSuperBytes = kSub_ * kTile;
    static constexpr int kSlots = 2;                       // TMA ring depth in sub-tiles
};
using ShapeB = TmaShape<3, 1, 5120, 2, 1, 8, 2>; // 3 CTAs / SM, 75 KB each: one staging buffer (default since round 2)
// Measured on the 1 GiB configs, kernel ms cfg2 / cfg3 (kv2-kv6, round 2), B against the shapes it replaced:
//   A = TmaShape<2, 2, 8192, 2> (2 CTAs / SM, 99 KB each, double-buffered staging; round 1) 0.395 / 0.346
//   B 0.391 / 0.342
//   H = TmaShape<2, 1, 7680, 2, 1, 12> (2 CTAs / SM x 12 worker warps: 48 KiB sub-tiles, 96 KiB per descriptor) 0.401 / 0.344
//   kSub = 4 (128 KiB per descriptor): 0.433 / 0.369 at 2 CTAs (36 pending mask registers), 0.539 / 0.453 at 3 (spills)
//   kSkew = 2: 0.391 / 0.347 at 2 CTAs, 0.423 / 0.366 at 3 (spills);  1 CTA x 16 worker warps: 0.436 / 0.367
//   look-back windows of 64 / 128 descriptors: 0.401 / 0.351 and 0.427 / 0.372;  re-polling one descriptor instead
//   of the window: no change.
// Just-in-time tickets (the producer draws the ticket of the next super-tile when the workers are half way through the
// compaction before it, not when a ring slot frees): B 0.374 / 0.337 (0.96 / 0.72 of the copy peak), A unchanged;
// signalled right after the prefix wait instead 0.377 / 0.341, after the whole compaction 0.402 / 0.351.  On top of it:
// no skew (compaction right after classification) 0.437 / 0.395; one 32 KiB sub-tile per descriptor 0.449 / 0.384.
// Two instruction-level variants on top of that changed nothing on cfg3 (kv12): the copy-out with one 32-bit add per
// entry (0.336 vs 0.336 ms; 0.388 vs 0.379 on cfg2) and the transpose's right shifts issued to the FMA pipe through
// __umulhi (0.337 vs 0.336) -- the quote-heavy case is not bound by the ALU pipe or by the copy-out's instruction count.
// With every look-back answered on its first poll (the descriptors of a previous build of the same bytes left in place:
// CSVB200_TUNE bit 0x400, a timing experiment) B runs 0.363 / 0.306 ms: the chain costs 7 % / 11 %, it is the
// workers waiting for their prefix (ncu: 11.7 % of the samples on that wait against 1.2 %), and none of the above
// moved it -- the wait follows the slowest of the ~440 tiles in flight, not the window, skew or descriptor size.
// (Tried and dropped: a ring of three 16 KiB half-stages shared by two warp groups, to fit double-buffered staging
//  into 70 KB.  It is NOT sound: the groups alternate on a slot, one group can run a whole phase ahead of the other,
//  and a parity wait cannot express that; it read stale data on the 1 GiB inputs.)

template <int kSub, int kWorkerWarps>
struct PrefixInfo {
    uint32_t pin[kSub];    // quote parity entering each sub-tile
    uint32_t cnt[kSub];    // entries each sub-tile emits (under its actual entry parity)
    uint64_t base[kSub];   // entries emitted before each sub-tile
    WarpState ws[kSub][kWorkerWarps];
};

template <class S>
struct __align__(1024) SmemTma {
    uint8_t in[S::kSlots][S::kTile];                 // TMA destinations, 1024-byte aligned (SWIZZLE_128B)
    uint16_t stage[S::kStageBufs][S::kStageCap + 8];   // 16-bit sub-tile-relative offsets
    uint64_t full[S::kSlots];               // producer -> workers (TMA complete_tx)
    uint64_t empty[S::kSlots];              // workers -> producer
    uint64_t agg_full[S::kRing];               // workers -> look-back warp
    uint64_t pref_full[S::kRing];              // look-back warp -> workers
    uint64_t go;                               // workers -> producer: "half way through this iteration's compaction"
    uint32_t tile_id[S::kSlots];            // super-tile id of the part in each slot
    uint32_t agg_tile[S::kRing];
    uint32_t warp_agg[S::kRing][S::kSub][S::kWorkers];
    // CSVB200_BUILD_VALIDATE: per warp {newlines if entered outside quotes [15:0], newlines in all [30:16], any byte >= 0x80 [31]}
    uint32_t warp_nl[S::kRing][S::kSub][S::kWorkers];
    PrefixInfo<S::kSub, S::kWorkers> pref[S::kRing];
};

// three CTAs per SM: 3 x (dynamic + 1 KiB reserved per CTA) must fit the SM's 228 KiB
static_assert(sizeof(SmemTma<ShapeB>) <= 75 * 1024, "3 CTAs / SM need <= 75 KiB each");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// try_wait suspends the warp in hardware up to the time hint instead of burning issue slots
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    const uint32_t addr = smem_u32(bar);
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(addr), "r"(parity), "r"(2000u)
            : "memory");
    } while (!ok);
}
// (ptxas turns try_wait into a SYNCS.TRYWAIT + NANOSLEEP.SYNCS loop that comes back every ~12 ns: the two service warps,
// which wait for most of a super-tile period, execute 50 M of the kernel's 300 M warp instructions that way (ncu, round
// 2).  Sleeping 64 / 128 / 256 ns after a failed try -- look-back warp alone or the producer too -- changed nothing:
// 0.3765 / 0.3410 ms against 0.3758-0.3764 / 0.3405-0.3420, profiles/r02_kvariants.md kv13: the spinning warps only take
// issue slots nobody else wants.)
__device__ __forceinline__ void tma_load_tile(void* smem_dst, const CUtensorMap* tmap, int32_t c0, int32_t c1, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
template <class S>
__device__ __forceinline__ void worker_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(S::kWorkerThreads) : "memory"); }

// streams staged entries [j0, j1) (staging indices, j0 even) of a run whose staging index 0 maps to
// global slot gbase; positions are tile_pos + 16-bit offset
template <class S>
__device__ __forceinline__ void copy_out_range(const BuildParams& p, const uint16_t* stg, uint32_t local0, uint32_t j0,
                                               uint32_t j1, uint64_t gbase, uint64_t tile_pos, uint32_t tid)
{
    uint64_t* out = p.index + gbase;
    if (gbase + j1 <= p.cap) {
        const uint32_t j1e = j1 & ~1u;
        // (Splitting tile_pos into a shared high word and one 32-bit add per entry halves this loop's instructions
        //  (11 -> 5 per store) and measured SLOWER twice, 0.416 vs 0.400 ms: the stores then leave in bursts that
        //  collide with the TMA reads; the paced version interleaves better with them.)
        for (uint32_t j = j0 + 2u * tid; j < j1e; j += 2u * S::kWorkerThreads) {
            const uint32_t pr = *reinterpret_cast<const uint32_t*>(&stg[j - local0]);
            stg_128(out + j, tile_pos + (pr & 0xffffu), tile_pos + (pr >> 16));
        }
        if ((j1 & 1u) && tid == 0 && j1 > j0) out[j1 - 1] = tile_pos + stg[j1 - 1 - local0];
    } else {
        for (uint32_t j = j0 + tid; j < j1; j += S::kWorkerThreads)
            if (gbase + j < p.cap) out[j] = tile_pos + stg[j - local0];
    }
}

// per-thread state of a classified sub-tile awaiting compaction
struct TileRegs {
    uint32_t s[kGroups];   // separator masks
    uint32_t x[kGroups];   // in-string masks relative to the warp start
    uint32_t exc;          // packed exclusive warp scan: entries before this thread (outside-hypothesis | total << 16)
};
template <int kSub>
struct SuperRegs {
    TileRegs sub[kSub];
    uint32_t tile;         // super-tile id
};

// Ordered compaction of one sub-tile: expand the masks into 16-bit offsets in shared memory at the
// scanned slots, then stream the run out as 16-byte stores.  `seq` numbers the sub-tile compactions
// of this CTA (it alternates the staging buffer when there are two).
template <class S>
__device__ __forceinline__ void compact_sub(SmemTma<S>& sm, const BuildParams& p, const TileRegs& t, const PrefixInfo<S::kSub, S::kWorkers>& pi,
                                            int sub, uint32_t super_tile, uint32_t seq, uint32_t tid, uint32_t warp)
{
    constexpr uint32_t kCap = (uint32_t)S::kStageCap;
    const uint32_t pin = pi.pin[sub];
    const uint32_t cnt = pi.cnt[sub];
    const uint64_t g0 = p.out_base + pi.base[sub];   // slot of the sub-tile's first entry
    const uint32_t head = (uint32_t)(g0 & 1ull);      // keep even slots on even staging indices
    const uint32_t end = cnt + head;
    const uint64_t gbase = g0 - head;
    const uint64_t tile_pos = p.pos_bias + (uint64_t)super_tile * S::kSuperBytes + (uint64_t)sub * S::kTile;
    const WarpState ws = pi.ws[sub][warp];
    const uint32_t h = pin ^ ws.par;                  // parity entering this warp
    const uint32_t ex_a0 = t.exc & 0xffffu, ex_tt = t.exc >> 16;
    const uint32_t slot0 = head + (pin ? ws.off1 : ws.off0) + (h ? ex_tt - ex_a0 : ex_a0);
    const uint32_t flip = 0u - h;
    uint16_t* stg = sm.stage[S::kStageBufs == 2 ? (seq & 1u) : 0u];
    // one staging buffer: the copy-out of the previous sub-tile must be over before it is written again
    // (with two buffers the other buffer's barrier already orders this)
    if (S::kStageBufs == 1) worker_barrier<S>();
    if (end <= kCap) {
        uint16_t* dst = stg + slot0;
        const bool sparse = cnt < 3u * (uint32_t)(S::kTile / 32);   // fewer than 3 entries per 32-byte group on average
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            uint32_t m = t.s[g] & ~(t.x[g] ^ flip);   // structure = all_struct & !string_mask (avx/stage1.rs:400-406)
            const uint32_t rel0 = tid * kBytesPerThread + 32u * g;
            const uint32_t c = (uint32_t)__popc(m);
            // two entries per trip: immediate store offsets, one pointer bump, half the branches
            // (0.396 vs 0.403 ms on cfg2 against a one-entry loop; walking two groups per loop for more ILP
            //  measured slower, 0.439 ms: this phase is issue-bound)
            if (S::kExpand == 2 && sparse) {
                uint16_t* d = dst;
#pragma unroll 1
                for (; m; d += 2) {
                    d[0] = (uint16_t)(rel0 + (uint32_t)__ffs((int)m) - 1u);
                    m &= m - 1u;
                    if (m) d[1] = (uint16_t)(rel0 + (uint32_t)__ffs((int)m) - 1u);
                    m &= m - 1u;
                }
                dst += c;
                continue;
            }
#pragma unroll 1
            for (uint32_t k = 0; k + 1u < c; k += 2u) {
                const uint32_t b0 = (uint32_t)__ffs((int)m) - 1u;
                m &= m - 1u;   // blsr (stage1.rs:239)
                const uint32_t b1 = (uint32_t)__ffs((int)m) - 1u;
                m &= m - 1u;
                dst[0] = (uint16_t)(rel0 + b0);
                dst[1] = (uint16_t)(rel0 + b1);
                dst += 2;
            }
            if (c & 1u) *dst++ = (uint16_t)(rel0 + (uint32_t)__ffs((int)m) - 1u);
        }
        worker_barrier<S>();
        if (head && tid == 0 && cnt > 0 && g0 < p.cap) p.index[g0] = tile_pos + stg[1];
        copy_out_range<S>(p, stg, 0u, 2u * head, end, gbase, tile_pos, tid);
        // no trailing barrier: see above
    } else {
        // dense sub-tile (more than kStageCap entries): several staging rounds
        for (uint32_t r0 = 0; r0 < end; r0 += kCap) {
            uint32_t slot = slot0;
#pragma unroll
            for (int g = 0; g < kGroups; ++g) {
                uint32_t m = t.s[g] & ~(t.x[g] ^ flip);
                const uint32_t rel0 = tid * kBytesPerThread + 32u * g;
                while (m) {
                    if (slot - r0 < kCap) stg[slot - r0] = (uint16_t)(rel0 + (uint32_t)__ffs((int)m) - 1u);
                    ++slot;
                    m &= m - 1u;
                }
            }
            worker_barrier<S>();
            const uint32_t r1 = min(end, r0 + kCap);
            if (r0 == 0 && head && tid == 0 && cnt > 0 && g0 < p.cap) p.index[g0] = tile_pos + stg[1];
            copy_out_range<S>(p, stg, r0, r0 == 0 ? 2u * head : r0, r1, gbase, tile_pos, tid);
            worker_barrier<S>();
        }
    }
}

__device__ __forceinline__ uint64_t dbg_clock()
{
    uint64_t c;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(c));
    return c;
}
__device__ __forceinline__ uint64_t dbg_globaltimer()
{
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// compaction of the `it`-th super-tile this CTA processed; every warp arrives on the producer's `go` barrier after the
// first sub-tile's compaction (see the producer)
template <class S, bool kDbg = false>
__device__ __forceinline__ void compact_super(SmemTma<S>& sm, const BuildParams& p, const SuperRegs<S::kSub>& t, uint32_t it,
                                              uint32_t tid, uint32_t warp)
{
    const uint32_t pb = it % S::kRing;
    if (kDbg && tid == 0) p.dbg[(uint64_t)t.tile * 8 + 2] = dbg_clock();      // the workers need the prefix from here
    mbar_wait(&sm.pref_full[pb], (it / S::kRing) & 1u);
    if (kDbg && tid == 0) p.dbg[(uint64_t)t.tile * 8 + 3] = dbg_clock();      // ... and have it here
    const PrefixInfo<S::kSub, S::kWorkers>& pi = sm.pref[pb];
#pragma unroll
    for (int sub = 0; sub < S::kSub; ++sub) {
        compact_sub<S>(sm, p, t.sub[sub], pi, sub, t.tile, it * S::kSub + sub, tid, warp);
        if (sub == 0 && (tid & 31u) == 0u) mbar_arrive(&sm.go);
    }
}

// kVal: CSVB200_BUILD_VALIDATE by-products; kEx: the cross-GPU exchange in the epilogue of the last CTA.  Both are
// compile-time so that the plain build keeps the register allocation it was tuned with (with the exchange code merely
// present the 64-register shape measured 0.401 instead of 0.391 ms on cfg2).
template <class S, bool kVal, bool kEx, bool kDbg = false>
__global__ void __launch_bounds__(S::kThreadsAll, S::kMinBlocks)
index_build_tma_kernel(const BuildParams p, const __grid_constant__ CUtensorMap tmap)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    SmemTma<S>& sm = *reinterpret_cast<SmemTma<S>*>(smem_raw);
    const uint32_t tid = threadIdx.x;
    const uint32_t lane = tid & 31u;
    const uint32_t warp = tid >> 5;
    constexpr int kSub = S::kSub, kSkew = S::kSkew, kRing = S::kRing, kWorkerWarps = S::kWorkers;

    if (p.run_flag != nullptr) {   // conditional redo
        if (p.pdl_wait == 2u) asm volatile("griddepcontrol.wait;" ::: "memory");   // launched under the build: its flag is final now
        if (*p.run_flag == 0u) return;                                              // ... and says it is not needed
    }
    // exchange form: the conditional redo behind this launch may be scheduled as soon as our CTAs leave
    if (kEx && tid == 0) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < S::kSlots; ++i) {
            mbar_init(&sm.full[i], 1);
            mbar_init(&sm.empty[i], kWorkerWarps);
        }
#pragma unroll
        for (int i = 0; i < kRing; ++i) {
            mbar_init(&sm.agg_full[i], kWorkerWarps);
            mbar_init(&sm.pref_full[i], 1);
        }
        mbar_init(&sm.go, kWorkerWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == S::kProducerWarp) {
        // ===== TMA producer: one elected lane =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmap)) : "memory");
            for (uint32_t it = 0;; ++it) {
                // Just-in-time ticket: the ticket of super-tile `it` is drawn when the workers are half way through the
                // compaction that precedes its classification (one sub-tile compaction ~ the TMA latency), not as soon
                // as a ring slot frees.  A ticket held for a whole period before its tile is classified makes every
                // later tile wait for an aggregate that is a period away -- and a CTA that waits for its prefix holds
                // such a ticket the whole time it waits.
                if (it > 0u) mbar_wait(&sm.go, (it - 1u) & 1u);
                // dynamic super-tile id: a tile only ever waits on tiles whose CTAs already hold a ticket.
                // (Taking the NEXT ticket early to hide the atomic's round trip measured slower, 0.423 vs
                // 0.418 ms: a ticket held for a whole super-tile period before its loads start delays the
                // look-back of every later tile.)
                uint32_t tile = atomicAdd(p.ticket, 1u);
                // every CTA takes tickets until it draws an invalid one: num_tiles + grid in all; the last one drawn
                // puts the counter back to zero for the next launch on this scratch
                if (tile == p.num_tiles + gridDim.x - 1u) *p.ticket = 0u;
                if (tile >= p.num_tiles) tile = kInvalidTile;
                if (kDbg && tile != kInvalidTile) p.dbg[(uint64_t)tile * 8 + 6] = dbg_clock();
#pragma unroll
                for (int sub = 0; sub < kSub; ++sub) {
                    const uint32_t sc = it * kSub + sub, st = sc % S::kSlots;
                    mbar_wait(&sm.empty[st], ((sc / S::kSlots) & 1u) ^ 1u);
                    sm.tile_id[st] = tile;
                    if (tile == kInvalidTile) {
                        mbar_arrive(&sm.full[st]);
                        break;   // the workers stop after an invalid sub-tile 0
                    }
                    mbar_arrive_expect_tx(&sm.full[st], (uint32_t)S::kTile);
#pragma unroll
                    for (int bx = 0; bx < S::kBoxes; ++bx)
                        tma_load_tile(sm.in[st] + bx * (kBoxRows * 128), &tmap, 0,
                                      (int32_t)((tile * (uint32_t)kSub + sub) * (uint32_t)S::kRows + bx * kBoxRows), &sm.full[st]);
                }
                if (tile == kInvalidTile) break;
            }
        }
    } else if (warp == S::kLookbackWarp) {
        // ===== scan of warp aggregates + decoupled look-back =====
        uint64_t cta_total = 0ull;   // separators (inside + outside quotes) of this CTA's super-tiles (lane 0)
        uint64_t cta_nl = 0ull;      // (validate) newlines outside quotes of this CTA's super-tiles
        uint32_t cta_hi = 0u;        // (validate) a byte >= 0x80 was seen
        for (uint32_t it = 0;; ++it) {
            const uint32_t b = it % kRing;
            mbar_wait(&sm.agg_full[b], (it / kRing) & 1u);
            const uint32_t tile = sm.agg_tile[b];
            if (tile == kInvalidTile) break;
            if (kDbg && lane == 0) {
                uint32_t smid;
                asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
                p.dbg[(uint64_t)tile * 8 + 0] = dbg_clock();                  // all aggregates of the super-tile are in
                p.dbg[(uint64_t)tile * 8 + 4] = (uint64_t)smid | ((uint64_t)blockIdx.x << 16) | ((uint64_t)it << 32);
                p.dbg[(uint64_t)tile * 8 + 5] = dbg_globaltimer();
            }
            PrefixInfo<kSub, kWorkerWarps>& pi = sm.pref[b];
            // fold the kSub x 8 warp aggregates in file order; remember the state entering every warp
            // and the (parity, c0, c1) composite at every sub-tile boundary
            uint32_t par = 0u, o0 = 0u, o1 = 0u;
            uint32_t nl_a = 0u, nl_b = 0u, any_hi = 0u;   // newlines outside quotes if the super-tile is entered outside / inside
            uint32_t sub_par[kSub], sub_o0[kSub], sub_o1[kSub];
#pragma unroll
            for (int sub = 0; sub < kSub; ++sub) {
                sub_par[sub] = par;
                sub_o0[sub] = o0;
                sub_o1[sub] = o1;
#pragma unroll
                for (int w = 0; w < kWorkerWarps; ++w) {
                    const uint32_t v = sm.warp_agg[b][sub][w];
                    const uint32_t wa0 = v & 0x7fffu, wt = (v >> 16) & 0x7fffu, wa1 = wt - wa0;
                    if (lane == 0) {
                        // warp state relative to the start of ITS sub-tile
                        pi.ws[sub][w].par = par ^ sub_par[sub];
                        pi.ws[sub][w].off0 = (sub_par[sub] ? o1 : o0) - (sub_par[sub] ? sub_o1[sub] : sub_o0[sub]);
                        pi.ws[sub][w].off1 = (sub_par[sub] ? o0 : o1) - (sub_par[sub] ? sub_o0[sub] : sub_o1[sub]);
                    }
                    o0 += par ? wa1 : wa0;
                    o1 += par ? wa0 : wa1;
                    if (kVal) {
                        const uint32_t nv = sm.warp_nl[b][sub][w];
                        const uint32_t n0 = nv & 0xffffu, n1 = ((nv >> 16) & 0x7fffu) - n0;
                        nl_a += par ? n1 : n0;
                        nl_b += par ? n0 : n1;
                        any_hi |= nv >> 31;
                    }
                    par ^= v >> 31;
                }
            }
            if (lane == 0)
                st_relaxed_u64(p.desc + (uint64_t)tile * kDescStride,
                               kStatusAgg | ((uint64_t)p.desc_tag << kTagShift) | (par ? kParityBit : 0ull) | (uint64_t)o0 | ((uint64_t)o1 << 20));
            uint32_t pin;
            uint64_t base;
            // one 32-descriptor window per round trip (wider windows measured slower both rounds: 0.400 / 0.427 ms
            // for 64 / 128 on cfg2 against 0.395 -- more polling traffic on the same lines)
            decoupled_lookback<S::kLook, kDbg>(p, tile, lane, pin, base);
            if (kDbg && lane == 0) {
                p.dbg[(uint64_t)tile * 8 + 1] = dbg_clock();                  // the prefix is known
                p.dbg[(uint64_t)tile * 8 + 7] = dbg_globaltimer();
            }
            if (lane == 0) {
                const uint32_t pend = pin ^ par;
                const uint64_t cend = base + (pin ? o1 : o0);
                st_relaxed_u64(p.desc + (uint64_t)tile * kDescStride,
                               kStatusPrefix | ((uint64_t)p.desc_tag << kTagShift) | (pend ? kParityBit : 0ull) | (cend & kCountMask));
#pragma unroll
                for (int sub = 0; sub < kSub; ++sub) {
                    const uint64_t b0 = base + (pin ? sub_o1[sub] : sub_o0[sub]);
                    const uint64_t b1 = sub + 1 < kSub ? base + (pin ? sub_o1[sub + 1 < kSub ? sub + 1 : sub] : sub_o0[sub + 1 < kSub ? sub + 1 : sub])
                                                       : cend;
                    pi.pin[sub] = pin ^ sub_par[sub];
                    pi.base[sub] = b0;
                    pi.cnt[sub] = (uint32_t)(b1 - b0);
                }
                if (tile == p.num_tiles - 1) write_result(p, cend, pend);
                if (tile == 0u && p.write_sentinel && p.cap > 0) p.index[0] = 0ull;
                cta_total += (uint64_t)(o0 + o1);
                if (kVal) {
                    cta_nl += pin ? nl_b : nl_a;
                    if (any_hi) {
                        cta_hi = 1u;
                        atomicOr(p.nonascii_bitmap + (tile >> 5), 1u << (tile & 31u));
                    }
                }
                mbar_arrive(&sm.pref_full[b]);
            }
            __syncwarp();
        }
        if (lane == 0) {
            if (p.total_out != nullptr && cta_total != 0ull) atomicAdd(p.total_out, (unsigned long long)cta_total);
            if (kVal) {
                if (cta_nl != 0ull) atomicAdd(p.nl_out, (unsigned long long)cta_nl);
                if (cta_hi) atomicOr(p.hi_out, 1u);
            }
            if (kVal || kEx) exchange_if_last(p);
        }
    } else {
        // ===== workers =====
        const uint64_t full_rows = p.n >> 7;
        const uint32_t tail = (uint32_t)(p.n & 127u);
        // masks of the super-tiles that are classified but not yet compacted (kSkew of them, oldest first)
        SuperRegs<kSub> pend[kSkew > 0 ? kSkew : 1];
#pragma unroll
        for (int k = 0; k < (kSkew > 0 ? kSkew : 1); ++k) pend[k].tile = kInvalidTile;

        for (uint32_t it = 0;; ++it) {
            const uint32_t b = it % kRing;
            SuperRegs<kSub> cur;
            cur.tile = kInvalidTile;
#pragma unroll
            for (int sub = 0; sub < kSub; ++sub) {
                TileRegs& tr = cur.sub[sub];
                tr.exc = 0u;
#pragma unroll
                for (int g = 0; g < kGroups; ++g) tr.s[g] = tr.x[g] = 0u;
                if (sub > 0 && cur.tile == kInvalidTile) continue;   // the producer stops after an invalid sub-tile 0
                const uint32_t sc = it * kSub + sub, st = sc % S::kSlots;
                mbar_wait(&sm.full[st], (sc / S::kSlots) & 1u);
                const uint32_t tile = sm.tile_id[st];
                cur.tile = tile;
                if (tile == kInvalidTile) continue;

                uint8_t* in = sm.in[st];
                // the sub-row tail of the file is outside the tensor map: its owner patches it in
                if (tail != 0u && ((uint64_t)tile * kSub + sub) * S::kRows + tid == full_rows) {
                    for (uint32_t k = 0; k < tail; ++k) {
                        const uint32_t c = (uint32_t)kChunks * tid + (k >> 4);
                        in[16u * (c ^ ((c >> 3) & 7u)) + (k & 15u)] = p.in[full_rows * 128u + k];
                    }
                }
                // ---- classify: 128 contiguous bytes (one swizzle row) per thread ----
                uint32_t q[kGroups], nlm[kGroups], hi = 0u;
#pragma unroll
                for (int g = 0; g < kGroups; ++g) {
                    uint32_t w[8];
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const uint32_t c = (uint32_t)kChunks * tid + 2 * g + i;
                        const uint4 v = *reinterpret_cast<const uint4*>(in + 16u * (c ^ ((c >> 3) & 7u)));
                        w[4 * i + 0] = v.x;
                        w[4 * i + 1] = v.y;
                        w[4 * i + 2] = v.z;
                        w[4 * i + 3] = v.w;
                    }
                    if (kVal) {
                        const Masks32x m = classify32x(w);
                        q[g] = m.quote;
                        tr.s[g] = m.sep;
                        nlm[g] = m.nl;
                        hi |= m.hi;
                    } else {
                        const Masks32 m = classify32(w);
                        q[g] = m.quote;
                        tr.s[g] = m.sep;
                        nlm[g] = 0u;
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.empty[st]);  // slot can be refilled

                // ---- quote regions relative to the warp start (string_mask, avx/stage1.rs:397) ----
                uint32_t warp_par = 0u, anyq = 0u;
#pragma unroll
                for (int g = 0; g < kGroups; ++g) anyq |= q[g];
                if (__any_sync(0xffffffffu, anyq != 0u)) {
                    uint32_t carry = 0u;
#pragma unroll
                    for (int g = 0; g < kGroups; ++g) {
                        tr.x[g] = prefix_xor32(q[g]) ^ carry;
                        carry = 0u - (tr.x[g] >> 31);
                    }
                    const uint32_t bal = __ballot_sync(0xffffffffu, carry != 0u);
                    const uint32_t lane_in = __popc(bal & ((1u << lane) - 1u)) & 1u;
                    warp_par = __popc(bal) & 1u;
                    const uint32_t flip = 0u - lane_in;
#pragma unroll
                    for (int g = 0; g < kGroups; ++g) tr.x[g] ^= flip;
                }
                uint32_t a0 = 0u, tt = 0u;
#pragma unroll
                for (int g = 0; g < kGroups; ++g) {
                    a0 += __popc(tr.s[g] & ~tr.x[g]);
                    tt += __popc(tr.s[g]);
                }
                const uint32_t packed = a0 | (tt << 16);
                uint32_t inc = packed;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t v = __shfl_up_sync(0xffffffffu, inc, d);
                    if (lane >= (uint32_t)d) inc += v;
                }
                tr.exc = inc - packed;
                if (lane == 31) sm.warp_agg[b][sub][warp] = inc | (warp_par << 31);
                if (kVal) {
                    uint32_t n0 = 0u, nt = 0u;
#pragma unroll
                    for (int g = 0; g < kGroups; ++g) {
                        n0 += __popc(nlm[g] & ~tr.x[g]);
                        nt += __popc(nlm[g]);
                    }
                    const uint32_t nsum = __reduce_add_sync(0xffffffffu, n0 | (nt << 16));
                    const uint32_t anyhi = __any_sync(0xffffffffu, hi != 0u) ? 1u : 0u;
                    if (lane == 31) sm.warp_nl[b][sub][warp] = nsum | (anyhi << 31);
                }
            }
            if (lane == 31) {
                if (warp == 0) sm.agg_tile[b] = cur.tile;
                mbar_arrive(&sm.agg_full[b]);
            }

            if (kSkew == 0) {
                // no skew: the tile just classified is compacted at once (the other CTAs of the SM cover the look-back);
                // nothing outlives an iteration, which frees the registers the pending masks take
                if (cur.tile == kInvalidTile) break;
                compact_super<S, kDbg>(sm, p, cur, it, tid, warp);
                continue;
            }
            // ---- ordered compaction of the super-tile classified kSkew iterations ago: its look-back has
            //      had kSkew classify phases to complete ----
            if (pend[0].tile != kInvalidTile)
                compact_super<S, kDbg>(sm, p, pend[0], it - kSkew, tid, warp);
            else if (lane == 0u)
                mbar_arrive(&sm.go);   // nothing to compact yet: the producer may draw the next ticket at once
            if (cur.tile == kInvalidTile) {
                // drain: the younger pending super-tiles, oldest first (the producer has stopped: their arrivals on
                // `go` complete phases nobody waits for)
#pragma unroll
                for (int k = 1; k < kSkew; ++k)
                    if (pend[k].tile != kInvalidTile) compact_super<S, kDbg>(sm, p, pend[k], it - kSkew + k, tid, warp);
                break;
            }
#pragma unroll
            for (int k = 0; k + 1 < kSkew; ++k) pend[k] = pend[k + 1];
            pend[kSkew > 0 ? kSkew - 1 : 0] = cur;
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

}  // namespace

bool tma_path_usable(uint64_t n) { return n >= 8ull * kTileBytes && encode_tiled_fn() != nullptr; }

namespace {

// cudaFuncSetAttribute and the occupancy are properties of (kernel, device): cached per device ordinal
// (a second context on another GPU of the same process needs its own opt-in to > 48 KiB of shared memory)
constexpr int kMaxDevices = 64;
struct ShapeState {
    std::mutex mu;
    int grid_cap[kMaxDevices] = {};
};

template <class S, bool kVal = false, bool kEx = false, bool kDbg = false>
cudaError_t launch_shape(const BuildParams& p_in, cudaStream_t stream)
{
    static ShapeState state;
    BuildParams p = p_in;
    p.num_tiles = (uint32_t)((p.n + S::kSuperBytes - 1) / S::kSuperBytes);   // descriptors are per super-tile here
    if (p.num_tiles == 0) p.num_tiles = 1;
    EncodeTiledFn encode = encode_tiled_fn();
    if (!encode) return cudaErrorNotSupported;
    // 2-D view of the input: [rows = n / 128][128 bytes]; rows beyond the end read as zeros
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {128, (cuuint64_t)(p.n >> 7)};
    const cuuint64_t gstride[1] = {128};
    const cuuint32_t box[2] = {128, (cuuint32_t)kBoxRows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(p.in), gdim, gstride, box,
                              estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);   // (promotion NONE: no difference)
    if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
    int grid_cap;
    {
        std::lock_guard<std::mutex> lock(state.mu);
        if (state.grid_cap[dev] == 0) {
            e = cudaFuncSetAttribute(index_build_tma_kernel<S, kVal, kEx, kDbg>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)sizeof(SmemTma<S>));
            if (e != cudaSuccess) return e;
            cudaFuncSetAttribute(index_build_tma_kernel<S, kVal, kEx, kDbg>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 cudaSharedmemCarveoutMaxShared);
            int sms = 148, per_sm = 0;
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, index_build_tma_kernel<S, kVal, kEx, kDbg>, S::kThreadsAll,
                                                              sizeof(SmemTma<S>));
            if (e != cudaSuccess) return e;
            if (per_sm < 1) return cudaErrorLaunchOutOfResources;
            state.grid_cap[dev] = sms * per_sm;   // persistent: one resident CTA per slot
        }
        grid_cap = state.grid_cap[dev];
    }
    const unsigned grid = (unsigned)(p.num_tiles < (uint32_t)grid_cap ? p.num_tiles : (uint32_t)grid_cap);
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(S::kThreadsAll);
    cfg.dynamicSmemBytes = sizeof(SmemTma<S>);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = p.pdl_wait ? 1u : 0u;
    return cudaLaunchKernelEx(&cfg, index_build_tma_kernel<S, kVal, kEx, kDbg>, p, tmap);
}

}  // namespace

uint64_t build_flag_tile_bytes(bool use_tma) { return use_tma ? (uint64_t)ShapeB::kSuperBytes : (uint64_t)kTileBytes; }

cudaError_t launch_index_build_tma(const BuildParams& p, cudaStream_t stream)
{
    if (p.validate) return p.ex.peers ? launch_shape<ShapeB, true, true>(p, stream) : launch_shape<ShapeB, true, false>(p, stream);
    if (p.ex.peers) return launch_shape<ShapeB, false, true>(p, stream);
    if (p.dbg) return launch_shape<ShapeB, false, false, true>(p, stream);   // timeline instrumentation (tools/timeline.py)
    return launch_shape<ShapeB>(p, stream);
}

}  // namespace csvb200
