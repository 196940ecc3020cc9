// record_split.h -- which device materialises which records of a distributed index (csvb200_multi_materialize_columns).
// Pure host code with no CUDA dependency, so a CPU test can compile it with g++ alone.
//
// Segment k holds the global index slots [base[k], base[k + 1]) and its device holds byte shard k.  Record r (0 = first
// row after the header) reads the slots (r + 1) * jump ... (r + 2) * jump.  When all of them lie in one segment, every
// byte of the record lies in that segment's shard too: a field's bytes lie between two of its separators, and a
// separator's entry sits in the segment of the shard that holds it.  Such a record is INTERIOR to the segment and is
// materialised in place.  Any other live record is a BOUNDARY record: its slots run over two or more segments (more
// when a shard holds no separator at all), so it is staged on one device first.  There is at most one per cut.
//
// Record numbers are u32 and wrap, as in the kernels (materialize.cu field_range): the record after 0xFFFFFFFF is 0,
// and record 0xFFFFFFFF itself reads the header row's slots, since (r + 1) wraps to 0.
#pragma once
#include <algorithm>
#include <cstdint>
#include <vector>

namespace csvb200 {

struct RecordPiece {
    uint32_t first, count;    // records first, first + 1, ... (u32, wrapping), count of them
    uint32_t seg_lo, seg_hi;  // interior: seg_lo == seg_hi; boundary (count == 1): segments of its first and last slot;
                              // dead records ((r + 1) >= record_cnt: empty values, no slot is read): both == nseg
    bool interior() const { return seg_lo == seg_hi; }
};

// segment holding slot s (s < base[nseg]); empty segments (base[k] == base[k + 1]) hold nothing and are skipped
inline uint32_t segment_of(const uint64_t* base, uint32_t nseg, uint64_t s)
{
    return (uint32_t)(std::upper_bound(base, base + nseg + 1, s) - base) - 1;
}

// Splits nrec records from first_record on into pieces in record order, each record in exactly one piece.  Interior and
// dead runs are maximal; every boundary record is a piece of its own.
// base[0 .. nseg] is non-decreasing with base[0] = 0; jump >= 1; record_cnt * jump < base[nseg] (csvb200_multi_tape_init).
inline std::vector<RecordPiece> split_records(const uint64_t* base, uint32_t nseg, uint64_t jump, uint32_t record_cnt,
                                              uint32_t first_record, uint32_t nrec)
{
    std::vector<RecordPiece> out;
    for (uint64_t pos = 0; pos < nrec;) {
        const uint32_t r = (uint32_t)(first_record + pos);
        const uint32_t rp1 = r + 1u;
        const uint64_t left = nrec - pos;
        uint64_t count;
        if (rp1 >= record_cnt) {
            // dead up to the end of the window, or up to record 0xFFFFFFFF, which reads the header row
            count = record_cnt ? std::min<uint64_t>(left, 0xFFFFFFFFull - r) : left;
            out.push_back({r, (uint32_t)count, nseg, nseg});
        } else {
            const uint64_t lo = (uint64_t)rp1 * jump, hi = lo + jump;
            const uint32_t k = segment_of(base, nseg, lo);
            if (hi < base[k + 1]) {
                // the records of segment k run up to (r + 2) * jump <= base[k + 1] - 1, the live ones up to r + 1 < record_cnt
                const uint64_t last_rp1 = std::min<uint64_t>((base[k + 1] - 1) / jump - 1, record_cnt - 1u);
                count = std::min<uint64_t>(left, last_rp1 - rp1 + 1);
                out.push_back({r, (uint32_t)count, k, k});
            } else {
                count = 1;
                out.push_back({r, 1u, k, segment_of(base, nseg, hi)});
            }
        }
        pos += count;
    }
    return out;
}

}  // namespace csvb200
