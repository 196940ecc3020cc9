// validate.cu -- K7: ASCII / UTF-8 validation of the input (SURVEY 8f rank 4).
//
// The reference carries two validators that are not wired into the path: is_ascii (word-at-a-time,
// src/reader.rs:26-132, "Non-core") and a copied SIMD UTF-8 checker whose module line is commented out
// (src/avx/utf8check.rs, src/avx/mod.rs:3), while seek_record builds &str with from_utf8_unchecked
// (src/record_source.rs:97-101).  This kernel answers both questions in one HBM-bound pass:
//   is_ascii      = no byte >= 0x80                         (is_ascii's result)
//   valid_up_to   = what core::str::from_utf8 would report: the start of the first ill-formed
//                   sequence (UINT64_MAX when the whole input is well-formed UTF-8)
// Every well-formedness rule of UTF-8 is local to a 4-byte window, so each thread judges the
// sequences whose LEAD lies in its own 32 bytes with the bit-sliced rules of utf8slice.cuh (3 bytes of
// look-ahead, 3 of look-behind) and the answer is an atomicMin.  32-byte groups that are pure ASCII (the
// common case in CSV) cost two 128-bit loads and a mask test.
#include "internal.h"
#include "utf8_halo.h"
#include "utf8slice.cuh"

namespace csvb200 {

namespace {

__device__ __forceinline__ uint4 ldg_128(const void* p)
{
    uint4 r;
    asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// the 32-byte group starting at i0 (zero past the end of the input)
__device__ __forceinline__ void load_group(const uint8_t* __restrict__ in, uint64_t n, uint64_t i0, uint32_t w[8])
{
    if (i0 + 32 <= n) {
        const uint4 a = ldg_128(in + i0), b = ldg_128(in + i0 + 16);
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
        w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            uint32_t x = 0;
            for (int j = 0; j < 4; ++j)
                if (i0 + 4 * k + j < n) x |= (uint32_t)in[i0 + 4 * k + j] << (8 * j);
            w[k] = x;
        }
    }
}

// slow path of one group: halo bytes + the bit-sliced check (utf8slice.cuh); returns the absolute start of
// the first ill-formed sequence led from this group, or UINT64_MAX
__device__ __forceinline__ uint64_t judge_group(const uint8_t* __restrict__ in, uint64_t n, uint64_t i0, const uint32_t w[8])
{
    const uint32_t b1 = i0 >= 1 ? in[i0 - 1] : 0u, b2 = i0 >= 2 ? in[i0 - 2] : 0u, b3 = i0 >= 3 ? in[i0 - 3] : 0u;
    const uint32_t n0 = i0 + 32 < n ? in[i0 + 32] : 0x100u, n1 = i0 + 33 < n ? in[i0 + 33] : 0x100u,
                   n2 = i0 + 34 < n ? in[i0 + 34] : 0x100u;
    const uint32_t r = utf8_check32(w, utf8_owed(b1, b2, b3), n0, n1, n2);
    return r == kUtf8None ? UINT64_MAX : i0 + r;
}

// The same for one shard of a distributed input, global bytes [pos_bias, pos_bias + n), given its halo (utf8_halo.h).
// Only sequences LED inside the shard are judged: the after-halo is look-ahead only, since a lead there has its own
// look-ahead cut off by the halo's end and is judged by the device that holds it.  In the shard's last group the
// after-halo bytes take the places of the zero fill past n.  Returns the global start or UINT64_MAX.
__device__ __forceinline__ uint64_t judge_group_seg(const uint8_t* __restrict__ in, uint64_t n, uint64_t i0, const uint32_t w_in[8],
                                                    const Utf8Halo& h, uint64_t pos_bias)
{
    uint32_t w[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) w[k] = w_in[k];
    if (i0 + 32 > n) {
        const uint32_t a = h.after_len ? h.after & (0xffffffu >> (8 * (3 - h.after_len))) : 0u;
        const int at = 8 * (int)(n - i0);                              // bit position of byte n inside the group
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int sh = at - 32 * k;
            if (sh >= 0 && sh < 32) w[k] |= a << sh;
            else if (sh < 0 && sh > -24) w[k] |= a >> -sh;
        }
    }
    const uint32_t b1 = i0 ? in[i0 - 1] : h.before & 0xffu, b2 = i0 ? in[i0 - 2] : (h.before >> 8) & 0xffu,
                   b3 = i0 ? in[i0 - 3] : h.before >> 16;             // i0 is 0 or >= 32
    uint32_t nx[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const uint64_t q = i0 + 32 + d;
        nx[d] = q < n ? (uint32_t)in[q] : q - n < h.after_len ? (h.after >> (8 * (q - n))) & 0xffu : 0x100u;
    }
    const uint32_t r = utf8_check32(w, utf8_owed(b1, b2, b3), nx[0], nx[1], nx[2]);
    return r == kUtf8None || i0 + r >= n ? UINT64_MAX : pos_bias + i0 + r;
}

// kSeg: the shard form (utf8_validate_segment_kernel); the one-GPU kernel instantiates the code it always had
template <bool kSeg>
__device__ __forceinline__ void utf8_validate_body(const uint8_t* __restrict__ in, uint64_t n, uint64_t* __restrict__ result,
                                                   const Utf8Halo& h, uint64_t pos_bias)
{
    const uint64_t ngroups = (n + 31) / 32;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t bad = UINT64_MAX;
    uint32_t nonascii = 0u;
    // two groups per iteration: four 128-bit loads in flight per thread
    for (uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += 2 * stride) {
        uint32_t wa[8], wb[8];
        const uint64_t ia = 32 * g, ib = 32 * (g + stride);
        const bool has_b = g + stride < ngroups;
        load_group(in, n, ia, wa);
        if (has_b) load_group(in, n, ib, wb);
        uint32_t oa = 0u, ob = 0u;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            oa |= wa[k];
            ob |= has_b ? wb[k] : 0u;
        }
        // pure-ASCII groups (the common case in CSV) lead no multi-byte sequence; the zero fill past n keeps a shard's
        // after-halo out of oa / ob
        if (oa & 0x80808080u) {
            nonascii = 1u;
            const uint64_t r = kSeg ? judge_group_seg(in, n, ia, wa, h, pos_bias) : judge_group(in, n, ia, wa);
            bad = r < bad ? r : bad;
        }
        if (ob & 0x80808080u) {
            nonascii = 1u;
            const uint64_t r = kSeg ? judge_group_seg(in, n, ib, wb, h, pos_bias) : judge_group(in, n, ib, wb);
            bad = r < bad ? r : bad;
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const uint64_t o = __shfl_xor_sync(0xffffffffu, bad, d);
        bad = o < bad ? o : bad;
    }
    const uint32_t any = __ballot_sync(0xffffffffu, nonascii != 0u);
    if ((threadIdx.x & 31u) == 0u) {
        if (bad != UINT64_MAX) atomicMin(reinterpret_cast<unsigned long long*>(result), (unsigned long long)bad);
        if (any) atomicOr(reinterpret_cast<unsigned long long*>(result + 1), 1ull);
    }
}

__global__ void __launch_bounds__(256) utf8_validate_kernel(const uint8_t* __restrict__ in, uint64_t n,
                                                            uint64_t* __restrict__ result)   // {valid_up_to, non-ascii flag}
{
    utf8_validate_body<false>(in, n, result, Utf8Halo{0u, 0u, 0u}, 0);
}

__global__ void __launch_bounds__(256) utf8_validate_segment_kernel(const uint8_t* __restrict__ in, uint64_t n,
                                                                    uint64_t pos_bias, const Utf8Halo halo,
                                                                    uint64_t* __restrict__ result)
{
    utf8_validate_body<true>(in, n, result, halo, pos_bias);
}

// Only the tiles the build kernel flagged (a byte >= 0x80 somewhere inside): one CTA per flagged tile at a time.
// A tile that is not flagged is pure ASCII, so it neither leads a multi-byte sequence nor owes continuation bytes to
// a flagged neighbour's look-behind / look-ahead -- judging the flagged tiles alone gives from_utf8's answer.
__global__ void __launch_bounds__(256) utf8_validate_flagged_kernel(const uint8_t* __restrict__ in, uint64_t n,
                                                                    const uint32_t* __restrict__ bitmap, uint64_t tile_bytes,
                                                                    uint64_t* __restrict__ result)
{
    const uint64_t ntiles = (n + tile_bytes - 1) / tile_bytes;
    const uint64_t groups_per_tile = tile_bytes / 32;
    uint64_t bad = UINT64_MAX;
    for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        if (!((bitmap[t >> 5] >> (t & 31u)) & 1u)) continue;
        for (uint64_t k = threadIdx.x; k < groups_per_tile; k += blockDim.x) {
            const uint64_t i0 = t * tile_bytes + 32 * k;
            if (i0 >= n) break;
            uint32_t w[8];
            load_group(in, n, i0, w);
            uint32_t o = 0u;
#pragma unroll
            for (int j = 0; j < 8; ++j) o |= w[j];
            if (o & 0x80808080u) {
                const uint64_t r = judge_group(in, n, i0, w);
                bad = r < bad ? r : bad;
            }
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const uint64_t o = __shfl_xor_sync(0xffffffffu, bad, d);
        bad = o < bad ? o : bad;
    }
    if ((threadIdx.x & 31u) == 0u && bad != UINT64_MAX)
        atomicMin(reinterpret_cast<unsigned long long*>(result), (unsigned long long)bad);
}

}  // namespace

cudaError_t launch_utf8_validate_flagged(const uint8_t* in, uint64_t n, const uint32_t* bitmap, uint64_t tile_bytes,
                                         uint64_t* result, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint64_t blocks = (n + tile_bytes - 1) / tile_bytes;
    const uint64_t max_blocks = (uint64_t)sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    utf8_validate_flagged_kernel<<<(unsigned)blocks, 256, 0, stream>>>(in, n, bitmap, tile_bytes, result);
    return cudaGetLastError();
}

// two 32-byte groups per thread and sweep, at most 8 blocks per SM
static unsigned utf8_validate_blocks(uint64_t n)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint64_t blocks = ((n + 31) / 32 + 511) / 512;
    const uint64_t max_blocks = (uint64_t)sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    return (unsigned)blocks;
}

cudaError_t launch_utf8_validate(const uint8_t* in, uint64_t n, uint64_t* result, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    utf8_validate_kernel<<<utf8_validate_blocks(n), 256, 0, stream>>>(in, n, result);
    return cudaGetLastError();
}

cudaError_t launch_utf8_validate_segment(const uint8_t* in, uint64_t n, uint64_t pos_bias, const Utf8Halo& halo,
                                         uint64_t* result, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    utf8_validate_segment_kernel<<<utf8_validate_blocks(n), 256, 0, stream>>>(in, n, pos_bias, halo, result);
    return cudaGetLastError();
}

}  // namespace csvb200
