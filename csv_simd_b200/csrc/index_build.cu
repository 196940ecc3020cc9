// index_build.cu -- fused single-pass CSV structural index build for sm_100a.
//
// Replaces, in ONE kernel and one pass over the input (traffic = N + 8E):
//   reader::read            src/reader.rs:150-306      (64-byte block loop, tail padding, carries)
//   SimdInput::structure    src/avx/stage1.rs:193-407  (classify, bit-pack, clmul prefix-XOR, carry, mask)
//   Stage1::crush_set_bits  src/stage1.rs:162-296      (tzcnt/blsr extraction into the growing Vec<usize>)
//
// The two serial dependencies of the reference loop -- the 1-bit `inside_str`
// carry (reader.rs:218, stage1.rs:397,407) and the running `array_idx`
// (reader.rs:217, stage1.rs:176-177,292) -- become ONE decoupled look-back over
// the monoid (p, c0, c1):
//   p  = quote parity of a tile
//   c0 = number of separators outside quotes if the tile is entered outside quotes
//   c1 = the same if the tile is entered inside quotes
//   (p1,a0,a1) o (p2,b0,b1) = (p1^p2, a0 + (p1 ? b1 : b0), a1 + (p1 ? b0 : b1))
// so every tile learns both its carry-in parity and its output base from the
// same chain and the input is read exactly once.
//
// Per tile (32 KiB, 256 threads x 128 B):
//   1. coalesced 128-bit loads -> shared memory in the TMA SWIZZLE_128B pattern,
//      so each thread can read back its own 64 contiguous bytes conflict-free;
//   2. bit-sliced classification (bitslice.cuh) -> 32-bit quote / separator masks;
//   3. in-word prefix-XOR (shift-xor), thread parities via one ballot, packed
//      (c0 | total) warp scan with shuffles, 8-entry warp-aggregate scan;
//   4. warp-parallel decoupled look-back (single u64 descriptor per tile);
//   5. ordered compaction: every thread expands its mask into 16-bit tile-relative
//      offsets in shared memory at its scanned slot, then the CTA streams the tile's
//      run out as full 16-byte stores (2 entries) of pos_bias + tile_base + offset.
#include <mutex>

#include "index_common.cuh"

namespace csvb200 {

namespace {

// Shared memory (dynamic): the input tile is dead once every thread has pulled its bytes into
// registers, so the 16-bit staging area of the compaction (worst case one entry per byte, +8
// slots of slack for 16-byte store alignment) aliases it.
struct __align__(1024) Smem {
    union {
        uint8_t in[kTileBytes];
        uint16_t stage[kTileBytes + 8];
    };
    uint32_t warp_agg[kWarps];
    uint32_t warp_nl[kWarps];   // (validate) as in index_build_tma.cu
    WarpState warp_state[kWarps];
    uint32_t tile;
    uint32_t pin;
    uint32_t tot0, tot1;
    uint64_t base;
};

__global__ void __launch_bounds__(kThreads, 3) index_build_kernel(const BuildParams p)
{
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    const uint32_t tid = threadIdx.x;
    const uint32_t lane = tid & 31u;
    const uint32_t warp = tid >> 5;

    if (p.run_flag != nullptr && *p.run_flag == 0u) return;   // conditional redo that is not needed
    // dynamic tile id: a tile only ever waits on tiles whose CTAs already started
    if (tid == 0) {
        sm.tile = atomicAdd(p.ticket, 1u);
        if (sm.tile == p.num_tiles - 1u) *p.ticket = 0u;   // the last ticket: back to zero for the next launch
    }
    __syncthreads();
    const uint32_t tile = sm.tile;
    const uint64_t tile_off = (uint64_t)tile * kTileBytes;

    // ---- 1. global -> shared, coalesced, swizzled (chunk' = chunk ^ (row & 7), the TMA 128B swizzle) ----
    if (tile_off + kTileBytes <= p.n) {   // full tile: no bounds checks (all tiles but the last)
        uint4 v[kChunks];
#pragma unroll
        for (int i = 0; i < kChunks; ++i) v[i] = ldg_stream_128(p.in + tile_off + 16ull * (tid + kThreads * i));
#pragma unroll
        for (int i = 0; i < kChunks; ++i) {
            const uint32_t c = tid + kThreads * i;
            *reinterpret_cast<uint4*>(sm.in + 16u * (c ^ ((c >> 3) & 7u))) = v[i];
        }
    } else {
#pragma unroll 1
        for (int i = 0; i < kChunks; ++i) {
            const uint32_t c = tid + kThreads * i;
            const uint64_t goff = tile_off + 16ull * c;
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (goff + 16 <= p.n) {
                v = ldg_stream_128(p.in + goff);
            } else if (goff < p.n) {
                // the reference zero-pads the final block (avx/stage1.rs:54-57,64-88)
                const uint32_t rem = (uint32_t)(p.n - goff);
                uint32_t w0 = 0u, w1 = 0u, w2 = 0u, w3 = 0u;
                for (uint32_t b = 0; b < rem; ++b) {
                    const uint32_t byte = (uint32_t)p.in[goff + b] << (8 * (b & 3));
                    if (b < 4) w0 |= byte;
                    else if (b < 8) w1 |= byte;
                    else if (b < 12) w2 |= byte;
                    else w3 |= byte;
                }
                v = make_uint4(w0, w1, w2, w3);
            }
            *reinterpret_cast<uint4*>(sm.in + 16u * (c ^ ((c >> 3) & 7u))) = v;
        }
    }
    __syncthreads();

    // ---- 2. each thread: its 128 contiguous bytes (one swizzle row) -> quote / separator masks ----
    uint32_t q[kGroups], s[kGroups], nlm[kGroups], hi = 0u;
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
        uint32_t w[8];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const uint32_t c = (uint32_t)kChunks * tid + 2 * g + i;   // logical chunk; row = c >> 3
            const uint32_t pc = c ^ ((c >> 3) & 7u);
            const uint4 v = *reinterpret_cast<const uint4*>(sm.in + 16u * pc);
            w[4 * i + 0] = v.x;
            w[4 * i + 1] = v.y;
            w[4 * i + 2] = v.z;
            w[4 * i + 3] = v.w;
        }
        const Masks32x m = classify32x(w);
        q[g] = m.quote;
        s[g] = m.sep;
        nlm[g] = m.nl;
        hi |= m.hi;
    }

    // ---- 3. quote regions inside the warp (relative to the warp start) ----
    // x = inclusive prefix-XOR of the quote bits: opening quote bit = 1, closing = 0,
    // exactly the reference's string_mask (avx/stage1.rs:397).
    uint32_t x[kGroups];
    uint32_t warp_par = 0u, anyq = 0u;
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
        x[g] = 0u;
        anyq |= q[g];
    }
    if (__any_sync(0xffffffffu, anyq != 0u)) {
        uint32_t carry = 0u;
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            x[g] = prefix_xor32(q[g]) ^ carry;
            carry = 0u - (x[g] >> 31);
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, carry != 0u);
        const uint32_t lane_in = __popc(bal & ((1u << lane) - 1u)) & 1u;
        warp_par = __popc(bal) & 1u;
        const uint32_t flip = 0u - lane_in;
#pragma unroll
        for (int g = 0; g < kGroups; ++g) x[g] ^= flip;
    }
    // counts under "warp entered outside quotes" (a0) and the hypothesis-free total (tt)
    uint32_t a0 = 0u, tt = 0u;
#pragma unroll
    for (int g = 0; g < kGroups; ++g) {
        a0 += __popc(s[g] & ~x[g]);
        tt += __popc(s[g]);
    }
    const uint32_t packed = a0 | (tt << 16);
    uint32_t inc = packed;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= (uint32_t)d) inc += v;
    }
    const uint32_t exc = inc - packed;
    if (lane == 31) sm.warp_agg[warp] = inc | (warp_par << 31);
    if (p.validate) {
        uint32_t n0 = 0u, nt = 0u;
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            n0 += __popc(nlm[g] & ~x[g]);
            nt += __popc(nlm[g]);
        }
        const uint32_t nsum = __reduce_add_sync(0xffffffffu, n0 | (nt << 16));
        const uint32_t anyhi = __any_sync(0xffffffffu, hi != 0u) ? 1u : 0u;
        if (lane == 31) sm.warp_nl[warp] = nsum | (anyhi << 31);
    }
    __syncthreads();  // also: every thread is done reading sm.in

    // ---- 4. warp 0: scan the 8 warp aggregates, publish, look back ----
    if (warp == 0) {
        uint32_t par = 0u, o0 = 0u, o1 = 0u;
        uint32_t nl_a = 0u, nl_b = 0u, any_hi = 0u;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            const uint32_t v = sm.warp_agg[w];
            const uint32_t wa0 = v & 0x7fffu, wt = (v >> 16) & 0x7fffu, wa1 = wt - wa0;
            if (lane == 0) {
                sm.warp_state[w].par = par;
                sm.warp_state[w].off0 = o0;
                sm.warp_state[w].off1 = o1;
            }
            o0 += par ? wa1 : wa0;
            o1 += par ? wa0 : wa1;
            if (p.validate) {
                const uint32_t nv = sm.warp_nl[w];
                const uint32_t n0 = nv & 0xffffu, n1 = ((nv >> 16) & 0x7fffu) - n0;
                nl_a += par ? n1 : n0;
                nl_b += par ? n0 : n1;
                any_hi |= nv >> 31;
            }
            par ^= v >> 31;
        }
        // (par, o0, o1) is the tile aggregate
        if (lane == 0)
            st_relaxed_u64(p.desc + (uint64_t)tile * kDescStride, kStatusAgg | ((uint64_t)p.desc_tag << kTagShift) | (par ? kParityBit : 0ull) | (uint64_t)o0 | ((uint64_t)o1 << 20));

        uint32_t pin;
        uint64_t base;
        decoupled_lookback<1>(p, tile, lane, pin, base);
        if (lane == 0) {
            const uint32_t pend = pin ^ par;
            const uint64_t cend = base + (pin ? o1 : o0);
            st_relaxed_u64(p.desc + (uint64_t)tile * kDescStride, kStatusPrefix | ((uint64_t)p.desc_tag << kTagShift) | (pend ? kParityBit : 0ull) | (cend & kCountMask));
            sm.pin = pin;
            sm.base = base;
            sm.tot0 = o0;
            sm.tot1 = o1;
            if (tile == p.num_tiles - 1) {
                write_result(p, cend, pend);
            }
            if (tile == 0u && p.write_sentinel && p.cap > 0) p.index[0] = 0ull;
            if (p.total_out != nullptr && (o0 | o1) != 0u) atomicAdd(p.total_out, (unsigned long long)(o0 + o1));
            if (p.validate) {
                const uint32_t nl = pin ? nl_b : nl_a;
                if (nl) atomicAdd(p.nl_out, (unsigned long long)nl);
                if (any_hi) {
                    atomicOr(p.hi_out, 1u);
                    atomicOr(p.nonascii_bitmap + (tile >> 5), 1u << (tile & 31u));
                }
            }
            exchange_if_last(p);
        }
    }
    __syncthreads();

    // ---- 5. ordered compaction ----
    const uint32_t pin = sm.pin;
    const uint64_t base = sm.base;
    const uint32_t cnt = pin ? sm.tot1 : sm.tot0;
    const uint64_t g0 = p.out_base + base;              // slot of this tile's first entry
    const uint32_t head = (uint32_t)(g0 & 1ull);         // keep even slots on even staging indices
    {
        const WarpState ws = sm.warp_state[warp];
        const uint32_t h = pin ^ ws.par;                 // parity entering this warp
        const uint32_t ex_a0 = exc & 0xffffu, ex_tt = exc >> 16;
        uint16_t* dst = sm.stage + head + (pin ? ws.off1 : ws.off0) + (h ? ex_tt - ex_a0 : ex_a0);
        const uint32_t flip = 0u - h;
#pragma unroll
        for (int g = 0; g < kGroups; ++g) {
            // structure = all_struct & !string_mask (avx/stage1.rs:400-406)
            uint32_t m = s[g] & ~(x[g] ^ flip);
            const uint32_t rel0 = tid * kBytesPerThread + 32u * g;
            while (m) {
                *dst++ = (uint16_t)(rel0 + (uint32_t)__ffs((int)m) - 1u);
                m &= m - 1u;  // blsr (stage1.rs:239)
            }
        }
    }
    __syncthreads();
    {
        const uint64_t tile_pos = p.pos_bias + tile_off;
        if (head && tid == 0 && cnt > 0 && g0 < p.cap) p.index[g0] = tile_pos + sm.stage[1];
        // staging index j = i + head is even for every pair, and g = g0 - head + j is even too
        const uint32_t end = cnt + head;
        const uint64_t gbase = g0 - head;
        uint64_t* out = p.index + gbase;
        if (gbase + end <= p.cap) {
            // common case: the whole run fits; full 16-byte stores except possibly the last entry
            const uint32_t end2 = end & ~1u;
            for (uint32_t j = 2u * head + 2u * tid; j < end2; j += 2u * kThreads) {
                const uint32_t pr = *reinterpret_cast<const uint32_t*>(&sm.stage[j]);
                stg_128(out + j, tile_pos + (pr & 0xffffu), tile_pos + (pr >> 16));
            }
            if ((end & 1u) && tid == 0 && end > 2u * head) out[end - 1] = tile_pos + sm.stage[end - 1];
        } else {
            for (uint32_t j = 2u * head + tid; j < end; j += kThreads)
                if (gbase + j < p.cap) out[j] = tile_pos + sm.stage[j];
        }
    }
}

// ---- pass A of the multi-GPU protocol: quote parity of a byte range ----------
// Only the 1-bit parity has to be known before a shard can be indexed (the
// counts fall out of the build itself), so this pass is a pure streaming
// XOR-reduction: SWAR "byte == 0x22" flags are XOR-accumulated and popcounted once.
__global__ void __launch_bounds__(256) quote_parity_kernel(const uint8_t* __restrict__ in, uint64_t n,
                                                           uint32_t* __restrict__ out)
{
    const uint64_t nvec = n / 16;
    uint32_t acc = 0u;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += stride) {
        const uint4 v = ldg_stream_128(in + 16 * i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t x = w[k] ^ 0x22222222u;
            // exact zero-byte test: bit 7 of every byte that equals zero
            acc ^= ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x | 0x7f7f7f7fu);
        }
    }
    uint32_t par = __popc(acc) & 1u;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (uint64_t b = nvec * 16; b < n; ++b) par ^= (in[b] == 0x22) ? 1u : 0u;
    }
    par = __reduce_xor_sync(0xffffffffu, par);
    __shared__ uint32_t s_par[8];
    if ((threadIdx.x & 31) == 0) s_par[threadIdx.x >> 5] = par;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t ^= s_par[w];
        if (t) atomicXor(out, 1u);
    }
}

// ---- speculative carry for the sharded build -----------------------------------------------------
// In RFC-4180-shaped data a quote whose neighbours are (delimiter, non-delimiter-non-quote) opens a
// field and one whose neighbours are (non-delimiter-non-quote, delimiter) closes one; quotes touching
// another quote ("" escapes, empty fields) and quotes between two delimiters are ambiguous and skipped.
// The first decisive quote in the shard's first `window` bytes fixes the parity entering the shard.
// This is only a PREDICTION: the build that uses it reports its end parity and the carry it used, the
// true carry chain is verified after the all-gather (verify_carry_kernel) and a wrong guess is rebuilt,
// so the result is exact for any input (the reference's toggle semantics, src/avx/stage1.rs:363-407,
// do not require well-formed CSV).
//
// One CTA of 1024 threads, 16 bytes per thread and round (16 KiB per round, coalesced 128-bit loads).
// cell = {0 (entry count entering the shard), predicted parity, 1 if a decisive quote was found, 0}.
constexpr int kPredictThreads = 1024;

__global__ void __launch_bounds__(kPredictThreads) predict_carry_kernel(const uint8_t* __restrict__ in, uint64_t n,
                                                                        uint64_t window, uint64_t* __restrict__ cell)
{
    __shared__ uint32_t s_warp[kPredictThreads / 32];
    __shared__ uint32_t s_res[3];   // found, predicted parity, running parity
    // the index build behind this launch may start now (programmatic dependent launch): only the threads that read
    // the cell wait for this grid to finish (BuildParams::pdl_wait)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint64_t lim = n < window ? n : window;
    uint32_t run_par = 0u, pred = 0u, found = 0u;
    for (uint64_t base = 0; base < lim; base += 16ull * kPredictThreads) {
        const uint64_t i0 = base + 16ull * tid;
        uint32_t qm = 0u, am = 0u, bm = 0u;
        if (i0 < lim) {
            uint8_t b[18];
            b[0] = i0 > 0 ? in[i0 - 1] : 0x22u;   // shard edges: treated as ambiguous
            if (i0 + 16 <= n) {
                const uint4 v = ldg_stream_128(in + i0);
                const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int k = 0; k < 16; ++k) b[1 + k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
            } else {
#pragma unroll
                for (int k = 0; k < 16; ++k) b[1 + k] = i0 + k < n ? in[i0 + k] : 0x22u;
            }
            b[17] = i0 + 16 < n ? in[i0 + 16] : 0x22u;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const uint32_t c = b[1 + k], prv = b[k], nxt = b[2 + k];
                const bool isq = c == 0x22u && i0 + k < lim;
                const bool dp = prv == 0x2Cu || prv == 0x0Du || prv == 0x0Au;
                const bool dn = nxt == 0x2Cu || nxt == 0x0Du || nxt == 0x0Au;
                const bool clean = isq && prv != 0x22u && nxt != 0x22u;
                qm |= (isq ? 1u : 0u) << k;
                am |= (clean && dp && !dn ? 1u : 0u) << k;   // opening
                bm |= (clean && !dp && dn ? 1u : 0u) << k;   // closing
            }
        }
        // thread: first decisive quote, quote parity before it, quote parity of the whole chunk
        const uint32_t dec = am | bm;
        const uint32_t f = dec ? (uint32_t)__ffs((int)dec) - 1u : 0u;
        const uint32_t t_before = __popc(qm & ((1u << f) - 1u)) & 1u;
        const uint32_t t_open = (am >> f) & 1u;
        const uint32_t t_par = __popc(qm) & 1u;
        // warp: nearest decisive lane
        const uint32_t bal = __ballot_sync(0xffffffffu, dec != 0u);
        const uint32_t pb = __ballot_sync(0xffffffffu, t_par != 0u);
        const uint32_t fl = bal ? (uint32_t)__ffs((int)bal) - 1u : 0u;
        const uint32_t w_before = (__popc(pb & ((1u << fl) - 1u)) & 1u) ^ __shfl_sync(0xffffffffu, t_before, (int)fl);
        const uint32_t w_open = __shfl_sync(0xffffffffu, t_open, (int)fl);
        if (lane == 0) s_warp[warp] = (bal ? 1u : 0u) | (w_open << 1) | (w_before << 2) | ((__popc(pb) & 1u) << 3);
        __syncthreads();
        if (tid == 0) {
            uint32_t acc = run_par, fnd = 0u, prd = 0u;
            for (int w = 0; w < kPredictThreads / 32; ++w) {
                const uint32_t v = s_warp[w];
                if (v & 1u) {
                    const uint32_t before = acc ^ ((v >> 2) & 1u);   // quotes in shard[0 .. i) mod 2
                    prd = ((v >> 1) & 1u) ? before : (before ^ 1u);
                    fnd = 1u;
                    break;
                }
                acc ^= (v >> 3) & 1u;
            }
            s_res[0] = fnd;
            s_res[1] = prd;
            s_res[2] = acc;
        }
        __syncthreads();
        found = s_res[0];
        pred = s_res[1];
        run_par = s_res[2];
        if (found) break;
        __syncthreads();
    }
    if (tid == 0) {
        cell[0] = 0ull;
        cell[1] = pred;
        cell[2] = found;
        cell[3] = 0ull;
    }
}

// After the all-gather of every rank's {entries emitted under the carry it used, end parity under that
// carry, carry used, total separators}: derive the TRUE carry of every shard (exclusive XOR-scan of
// the shard parities, shard parity = end ^ used) and, because flipping a shard's carry turns "outside"
// separators into "inside" ones and vice versa (c0 + c1 = total), the true entry count of every shard
// without another exchange.  cell <- {0, true carry of this rank, -, redo flag}; final[world][2]
// (optional) <- {true entry count, true carry} of every rank.
__global__ void verify_carry_kernel(const uint64_t* __restrict__ gathered, uint32_t world, uint32_t rank,
                                    uint64_t* __restrict__ cell, uint64_t* __restrict__ final_out)
{
    if (threadIdx.x != 0) return;
    uint32_t carry = 0u;
    for (uint32_t j = 0; j < world; ++j) {
        const uint64_t cnt = gathered[4 * j + 0], total = gathered[4 * j + 3];
        const uint32_t endp = (uint32_t)(gathered[4 * j + 1] & 1ull), used = (uint32_t)(gathered[4 * j + 2] & 1ull);
        if (final_out != nullptr) {
            final_out[2 * j + 0] = carry == used ? cnt : total - cnt;
            final_out[2 * j + 1] = carry;
        }
        if (j == rank) {
            cell[0] = 0ull;
            cell[1] = carry;
            cell[3] = carry != used ? 1ull : 0ull;
        }
        carry ^= endp ^ used;
    }
}

__global__ void exchange_kernel(const ExchangeArgs ex, const uint64_t* __restrict__ row4)
{
    if (threadIdx.x == 0) exchange_post_and_resolve(ex, row4[0], row4[1], row4[2], row4[3]);
}

// ---- K1 known-answer exports --------------------------------------------------
// quote_bits / all_struct words per 64-byte block, as get_struct_positions(16|3)
// returns them (avx/stage1.rs:392,394); bytes past n read as zero.
__global__ void block_masks_kernel(const uint8_t* __restrict__ in, uint64_t n, uint64_t* __restrict__ qw,
                                   uint64_t* __restrict__ sw)
{
    const uint64_t nblocks = (n + 63) / 64;
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        uint32_t v = 0;
        for (int k = 0; k < 4; ++k) {
            const uint64_t off = b * 64 + 4 * i + k;
            if (off < n) v |= (uint32_t)in[off] << (8 * k);
        }
        w[i] = v;
    }
    const Masks32 m0 = classify32(w), m1 = classify32(w + 8);
    qw[b] = (uint64_t)m0.quote | ((uint64_t)m1.quote << 32);
    sw[b] = (uint64_t)m0.sep | ((uint64_t)m1.sep << 32);
}

// class byte per input byte: the deprecated structure::run (src/structure.rs:10-58)
__global__ void class_bytes_kernel(const uint8_t* __restrict__ in, uint64_t n, uint8_t* __restrict__ out)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = class_byte(in[i]);
}

}  // namespace

cudaError_t launch_index_build(const BuildParams& p, cudaStream_t stream)
{
    if (p.num_tiles == 0) return cudaSuccess;
    // the opt-in to > 48 KiB of dynamic shared memory is per (kernel, device): cached per device ordinal
    static std::mutex mu;
    static bool configured[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return cudaErrorInvalidDevice;
    {
        std::lock_guard<std::mutex> lock(mu);
        if (!configured[dev]) {
            e = cudaFuncSetAttribute(index_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem));
            if (e != cudaSuccess) return e;
            configured[dev] = true;
        }
    }
    index_build_kernel<<<p.num_tiles, kThreads, sizeof(Smem), stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_quote_parity(const uint8_t* in, uint64_t n, uint32_t* out, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint64_t blocks = (n / 16 + 255) / 256;
    const uint64_t max_blocks = (uint64_t)sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    if (blocks == 0) blocks = 1;
    quote_parity_kernel<<<(unsigned)blocks, 256, 0, stream>>>(in, n, out);
    return cudaGetLastError();
}

cudaError_t launch_predict_carry(const uint8_t* in, uint64_t n, uint64_t window, uint64_t* cell, cudaStream_t stream)
{
    predict_carry_kernel<<<1, kPredictThreads, 0, stream>>>(in, n, window, cell);
    return cudaGetLastError();
}

cudaError_t launch_verify_carry(const uint64_t* gathered, uint32_t world, uint32_t rank, uint64_t* cell,
                                uint64_t* final_out, cudaStream_t stream)
{
    verify_carry_kernel<<<1, 32, 0, stream>>>(gathered, world, rank, cell, final_out);
    return cudaGetLastError();
}

cudaError_t launch_exchange(const ExchangeArgs& ex, const uint64_t* row4, cudaStream_t stream)
{
    exchange_kernel<<<1, 32, 0, stream>>>(ex, row4);
    return cudaGetLastError();
}

cudaError_t launch_block_masks(const uint8_t* in, uint64_t n, uint64_t* qw, uint64_t* sw, cudaStream_t stream)
{
    const uint64_t nblocks = (n + 63) / 64;
    if (nblocks == 0) return cudaSuccess;
    block_masks_kernel<<<(unsigned)((nblocks + 127) / 128), 128, 0, stream>>>(in, n, qw, sw);
    return cudaGetLastError();
}

cudaError_t launch_class_bytes(const uint8_t* in, uint64_t n, uint8_t* out, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    class_bytes_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(in, n, out);
    return cudaGetLastError();
}

}  // namespace csvb200
