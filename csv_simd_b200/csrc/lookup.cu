// lookup.cu -- K4: batched record / field lookups against a device-resident index.
//
// Replaces RecordSource::seek_record (src/record_source.rs:70-102) and
// RecordSource::seek_field (src/record_source.rs:104-140) for batches of
// independent queries.  One thread per query:
//   seek_field : None if r+1 >= record_cnt or f >= field_cnt;
//                s = (r+1)*row_size + f      (u32 arithmetic, as the reference);
//                start = index[s] + 1, end = index[s+1]
//   seek_record: None if r+1 >= record_cnt;
//                s = (r+1)*jump;  start = index[s] + 1, end = index[s + field_cnt]
// The (start, end) pair is written with one 16-byte store; None is
// (UINT64_MAX, UINT64_MAX).  A slot outside the index (where the reference
// would panic on the Vec bounds check) also yields None and bumps *oob.
// The access is a random 16-byte gather over a multi-GB index: HBM
// sector-bound, 40 algorithmic bytes per query (8 in, 16 gathered, 16 out).
#include "internal.h"

namespace csvb200 {

namespace {

// E: the entry type, u64 or the u32 of a compact index
template <class E>
__global__ void __launch_bounds__(256) seek_kernel(const LookupParams p)
{
    const E* __restrict__ index = static_cast<const E*>(p.index);
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; q < p.nq; q += stride) {
        const uint32_t r = p.rec[q];
        uint64_t start = UINT64_MAX, end = UINT64_MAX;
        bool live = (uint32_t)(r + 1u) < p.record_cnt;
        uint32_t s;
        uint64_t e_slot;
        if (p.fld != nullptr) {
            const uint32_t f = p.fld[q];
            live = live && f < p.field_cnt;
            s = (uint32_t)(r + 1u) * p.row_size + f;
            e_slot = (uint64_t)s + 1;
        } else {
            s = (uint32_t)(r + 1u) * p.row_size;
            e_slot = (uint64_t)s + p.field_cnt;
        }
        if (live) {
            if (e_slot < p.index_len) {
                start = ldg_entry(index + s) + 1;
                end = ldg_entry(index + e_slot);
            } else {
                atomicAdd(p.oob, 1u);
            }
        }
        asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(p.ranges + 2 * q), "l"(start), "l"(end) : "memory");
    }
}

// (sharded_entry, in internal.h, resolves a slot to the segment that holds it)
__global__ void __launch_bounds__(256) seek_sharded_kernel(const LookupParams p, const SegmentTable seg)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t q = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; q < p.nq; q += stride) {
        const uint32_t r = p.rec[q];
        uint64_t start = UINT64_MAX, end = UINT64_MAX;
        bool live = (uint32_t)(r + 1u) < p.record_cnt;
        uint32_t s;
        uint64_t e_slot;
        if (p.fld != nullptr) {
            const uint32_t f = p.fld[q];
            live = live && f < p.field_cnt;
            s = (uint32_t)(r + 1u) * p.row_size + f;     // u32 arithmetic, as the reference (src/record_source.rs:129)
            e_slot = (uint64_t)s + 1;
        } else {
            s = (uint32_t)(r + 1u) * p.row_size;         // src/record_source.rs:83
            e_slot = (uint64_t)s + p.field_cnt;
        }
        if (live) {
            if (e_slot < p.index_len) {
                start = sharded_entry(seg, s) + 1;
                end = sharded_entry(seg, e_slot);
            } else {
                atomicAdd(p.oob, 1u);
            }
        }
        asm volatile("st.global.v2.u64 [%0], {%1, %2};" ::"l"(p.ranges + 2 * q), "l"(start), "l"(end) : "memory");
    }
}

}  // namespace

cudaError_t launch_seek(const LookupParams& p, cudaStream_t stream)
{
    if (p.nq == 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint64_t blocks = (p.nq + 255) / 256;
    const uint64_t max_blocks = (uint64_t)sms * 32;
    if (blocks > max_blocks) blocks = max_blocks;
    if (p.entry_bytes == 4)
        seek_kernel<uint32_t><<<(unsigned)blocks, 256, 0, stream>>>(p);
    else
        seek_kernel<uint64_t><<<(unsigned)blocks, 256, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_seek_sharded(const LookupParams& p, const SegmentTable& seg, cudaStream_t stream)
{
    if (p.nq == 0) return cudaSuccess;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    uint64_t blocks = (p.nq + 255) / 256;
    const uint64_t max_blocks = (uint64_t)sms * 32;
    if (blocks > max_blocks) blocks = max_blocks;
    seek_sharded_kernel<<<(unsigned)blocks, 256, 0, stream>>>(p, seg);
    return cudaGetLastError();
}

}  // namespace csvb200
