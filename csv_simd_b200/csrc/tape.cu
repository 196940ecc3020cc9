// tape.cu -- K5: device-side Tape validation (SURVEY 8f rank 1).
//
// The reference accepts a file when (index.len() - 1) % jump == 0 (TapeCore::init, src/tape.rs:315-347)
// and otherwise returns InvalidCsvFormat without saying where the structure breaks; a file whose rows
// are ragged in a way that happens to cancel passes silently and every later seek_record / seek_field
// (src/record_source.rs:70-140) returns the wrong bytes.  This kernel checks what those seeks assume:
// entry s (s >= 1) of the index is the k-th separator of its record, k = (s - 1) % jump, so it must be
//   LF files   (jump = field_cnt)     : ',' for k < jump-1, CR or LF for k = jump-1
//   CRLF files (jump = field_cnt + 1) : ',' for k < jump-2, CR for k = jump-2, LF right after it for k = jump-1
// and reports the FIRST slot that is not (atomicMin), i.e. the first bad record.  HBM-bound: reads the
// index once (8E bytes, 4E for a compact index) and one byte per entry of the input (every 32-byte sector of a dense
// file: N).
#include "internal.h"

namespace csvb200 {

namespace {

// One row of 32 slots per warp step.  Everything that does not depend on the slot is hoisted: CRLF / LF is a
// template parameter, k = (s - 1) % jump lives in 32 bits and advances by 32 % jump, and the only 64-bit
// work left per slot is the position arithmetic (the first version spent ~100 instructions per slot row on
// 64-bit modulo / select chains and was issue-bound at 0.55 of the HBM peak).  E: the entry type, u64 or the u32 of a
// compact index.  kSeg: the segment form (one segment of a distributed index, see TapeValidateParams) -- its own
// instantiations, so the one-GPU ones compile to the code they always had.
template <bool kCrlf, class E, bool kSeg>
__global__ void __launch_bounds__(256) tape_validate_kernel(const TapeValidateParams p)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t jump = (uint32_t)p.jump;
    const uint32_t nl0 = jump - (kCrlf ? 2u : 1u);    // first line-end slot of a row (k >= nl0 is CR / LF territory)
    const uint64_t last = p.index_len - 1;            // slots are 1 .. last; i = s - 1 in [0, last)
    const uint64_t i_first = kSeg ? p.first_slot - 1 : 0;   // the segment form starts at its own first slot
    const uint32_t step = 32u % jump;                 // k advances by 32 slots per warp row
    const E* __restrict__ index = static_cast<const E*>(p.index) + 1;   // index[i] here is slot s = i + 1
    uint64_t bad = UINT64_MAX;                        // smallest failing i
    constexpr int kUnroll = 4;
    constexpr uint64_t kRun = 32 * 16;
    for (uint64_t run = i_first + warp0 * kRun; run < last; run += warps * kRun) {
        const uint64_t run_end = run + kRun < last ? run + kRun : last;
        uint32_t k = (uint32_t)((run + lane) % jump);
        for (uint64_t i = run + lane; i < run_end; i += 32 * kUnroll) {
            uint64_t pos[kUnroll];
            uint32_t byte[kUnroll], kk[kUnroll];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const uint64_t iu = i + 32ull * u;
                pos[u] = iu < run_end ? ldg_entry(index + iu) : UINT64_MAX;   // UINT64_MAX - bias >= n: treated as skipped below
                kk[u] = k;
                k += step;
                k = k >= jump ? k - jump : k;
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const uint64_t rel = pos[u] - p.pos_bias;
                byte[u] = rel < p.n ? (uint32_t)p.bytes[rel] : 0x100u;      // 0x100: no separator there (out of range)
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
                const uint64_t iu = i + 32ull * u;
                if (iu >= run_end) continue;
                const uint32_t b = byte[u];
                bool ok;
                if (kk[u] < nl0) {
                    ok = b == 0x2Cu;
                } else if (!kCrlf) {
                    ok = b == 0x0Au || b == 0x0Du;
                } else if (kk[u] == nl0) {
                    ok = b == 0x0Du;
                } else {
                    // the LF directly after its CR; a segment's first slot finds its CR's entry in prev_entry
                    ok = b == 0x0Au && (kSeg && iu == i_first ? p.prev_entry : ldg_entry(index + iu - 1)) + 1 == pos[u];
                }
                if (!ok && iu < bad) bad = iu;
            }
        }
    }
    // warp minimum, one atomic per warp that saw a violation
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        const uint64_t o = __shfl_xor_sync(0xffffffffu, bad, d);
        bad = o < bad ? o : bad;
    }
    if (lane == 0 && bad != UINT64_MAX)
        atomicMin(reinterpret_cast<unsigned long long*>(p.first_bad_slot), (unsigned long long)(bad + 1));
}

template <class E>
__global__ void gather_slots_kernel(const E* __restrict__ index, uint64_t index_len,
                                    const uint64_t* __restrict__ slots, uint64_t n, uint64_t* __restrict__ out)
{
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = slots[i] < index_len ? (uint64_t)index[slots[i]] : UINT64_MAX;
}

// four entries per thread and trip: one 16-byte load, two 16-byte stores (12 bytes of traffic per entry)
__global__ void __launch_bounds__(256) widen_entries_kernel(const uint32_t* __restrict__ in, uint64_t n,
                                                            uint64_t* __restrict__ out)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t n4 = n / 4;
    for (uint64_t i = t; i < n4; i += stride) {
        const uint4 v = reinterpret_cast<const uint4*>(in)[i];
        reinterpret_cast<ulonglong2*>(out)[2 * i] = make_ulonglong2(v.x, v.y);
        reinterpret_cast<ulonglong2*>(out)[2 * i + 1] = make_ulonglong2(v.z, v.w);
    }
    for (uint64_t i = 4 * n4 + t; i < n; i += stride) out[i] = in[i];
}

}  // namespace

cudaError_t launch_gather_slots(const void* index, uint32_t entry_bytes, uint64_t index_len, const uint64_t* slots,
                                uint64_t n, uint64_t* out, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    if (entry_bytes == 4)
        gather_slots_kernel<<<blocks, 128, 0, stream>>>(static_cast<const uint32_t*>(index), index_len, slots, n, out);
    else
        gather_slots_kernel<<<blocks, 128, 0, stream>>>(static_cast<const uint64_t*>(index), index_len, slots, n, out);
    return cudaGetLastError();
}

cudaError_t launch_widen_entries(const uint32_t* in, uint64_t n, uint64_t* out, cudaStream_t stream)
{
    if (n == 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint64_t blocks = (n / 4 + 255) / 256;
    const uint64_t max_blocks = (uint64_t)sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    if (blocks == 0) blocks = 1;
    widen_entries_kernel<<<(unsigned)blocks, 256, 0, stream>>>(in, n, out);
    return cudaGetLastError();
}

// blocks for `slots` slots: 8 warps per block, one run each, at most 8 blocks per SM
static unsigned tape_validate_blocks(uint64_t slots)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint64_t blocks = (slots + 32 * 16 * 8 - 1) / (32 * 16 * 8);
    const uint64_t max_blocks = (uint64_t)sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    if (blocks == 0) blocks = 1;
    return (unsigned)blocks;
}

cudaError_t launch_tape_validate(const TapeValidateParams& p, cudaStream_t stream)
{
    if (p.index_len <= 1 || p.jump == 0) return cudaSuccess;
    const unsigned blocks = tape_validate_blocks(p.index_len);
    if (p.jump > 0xffffffffull) return cudaErrorInvalidValue;
    const bool compact = p.entry_bytes == 4;
    if (p.crlf && compact)
        tape_validate_kernel<true, uint32_t, false><<<blocks, 256, 0, stream>>>(p);
    else if (p.crlf)
        tape_validate_kernel<true, uint64_t, false><<<blocks, 256, 0, stream>>>(p);
    else if (compact)
        tape_validate_kernel<false, uint32_t, false><<<blocks, 256, 0, stream>>>(p);
    else
        tape_validate_kernel<false, uint64_t, false><<<blocks, 256, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_tape_validate_segment(const TapeValidateParams& p, cudaStream_t stream)
{
    if (p.first_slot == 0 || p.first_slot >= p.index_len || p.jump == 0) return cudaSuccess;
    if (p.jump > 0xffffffffull) return cudaErrorInvalidValue;
    if (p.entry_bytes == 4) return cudaErrorInvalidValue;   // the segments of a distributed index hold u64 entries
    const unsigned blocks = tape_validate_blocks(p.index_len - p.first_slot);
    if (p.crlf)
        tape_validate_kernel<true, uint64_t, true><<<blocks, 256, 0, stream>>>(p);
    else
        tape_validate_kernel<false, uint64_t, true><<<blocks, 256, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace csvb200
