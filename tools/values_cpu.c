/* One-core CPU baseline of csvb200_seek_values over a host copy of the index: the scalar RecordSource::seek_field /
 * seek_record (two reads of the index per query) plus the copy of the raw value into a packed buffer, with the same
 * offsets and found bits.  Returns the checksum bench_values.py computes over the GPU's output.
 * Built at run time by tools/bench_values.py into a temporary directory. */
#include <stdint.h>
#include <string.h>

uint64_t values_cpu(const uint64_t* index, size_t index_len, const uint8_t* bytes, uint32_t record_cnt, uint32_t field_cnt,
                    uint32_t row_size, const uint32_t* rec, const uint32_t* fld, size_t nq, uint64_t* offsets, uint8_t* out,
                    uint64_t* found)
{
    uint64_t at = 0, sum = 0, nfound = 0;
    memset(found, 0, (nq + 63) / 64 * sizeof(uint64_t));
    for (size_t q = 0; q < nq; ++q) {
        offsets[q] = at;
        const uint32_t r = rec[q];
        if ((uint32_t)(r + 1u) >= record_cnt) continue;
        uint32_t s;
        uint64_t e;
        if (fld) {
            if (fld[q] >= field_cnt) continue;
            s = (uint32_t)(r + 1u) * row_size + fld[q];
            e = (uint64_t)s + 1;
        } else {
            s = (uint32_t)(r + 1u) * row_size;
            e = (uint64_t)s + field_cnt;
        }
        if (e >= index_len) continue;
        const uint64_t a = index[s] + 1, b = index[e];
        found[q / 64] |= 1ull << (q % 64);
        ++nfound;
        if (b <= a) continue;
        memcpy(out + at, bytes + a, b - a);
        at += b - a;
    }
    offsets[nq] = at;
    for (uint64_t i = 0; i < at; ++i) sum += out[i];
    return sum + 31u * at + 7u * nfound;
}
